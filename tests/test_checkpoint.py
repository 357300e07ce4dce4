"""Checkpoint compatibility (SURVEY §8 f.3), CPU only: reference-format files written by the UNMODIFIED reference
(util/misc.py save_model / auto_load_model, torch.optim.AdamW state) load into painter_b200 modules + FusedAdamW and
vice versa; the --finetune key filtering of main_train.py:199-224 drops and reports the same keys.

The reference side is tests/golden/ref_checkpoint.pt (`python -m oracle.make_golden checkpoint`): the file the
reference's save_model wrote, described key by key with a sha256 of every tensor, and the parameter names of each of
its lr_decay.param_groups_lrd groups.  The tests rebuild that file from its seeds and check it against the description
bit for bit before using it."""
import types
from functools import partial

import torch

from oracle import painter_oracle as po
from oracle.make_golden import CKPT_CFG, describe_checkpoint
from oracle.synth import synth_state_dict

from _common import load_golden

CFG = po.PainterConfig(**CKPT_CFG)


def _ours():
    from painter_b200 import models_painter
    m = models_painter.Painter(img_size=(64, 32), patch_size=16, embed_dim=64, depth=24, num_heads=1,
                               drop_path_rate=0.1, window_size=2, qkv_bias=True, mlp_ratio=4,
                               norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), window_block_indexes=[],
                               residual_block_indexes=[], use_rel_pos=True, decoder_embed_dim=64)
    return m


def _args(tmp_path, **kw):
    return types.SimpleNamespace(output_dir=str(tmp_path), resume="", auto_resume=True, start_epoch=0, **kw)


def _equal_sd(a, b):
    return a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)


def _scaler():
    """The loss scaler misc.NativeScalerWithGradNormCount wraps and whose state_dict it saves."""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # without a GPU it is created disabled
        return torch.amp.GradScaler("cuda")


def _reference_layout(gold, model):
    """torch.optim.AdamW over the reference's layer-decay groups of `model` (same parameter names per group, same
    lr_scale / weight_decay), lr 1e-3."""
    named = dict(model.named_parameters())
    saved = gold["checkpoint"]["optimizer"]["param_groups"]
    groups = [{"params": [named[n] for n in names], "lr_scale": g["lr_scale"], "weight_decay": g["weight_decay"]}
              for names, g in zip(gold["group_names"], saved)]
    return torch.optim.AdamW(groups, lr=1e-3)


def _load(path):
    return torch.load(path, map_location="cpu", weights_only=False)


def test_reference_checkpoint_resumes_into_painter_b200_and_back(tmp_path):
    from painter_b200 import checkpoint
    from painter_b200.optim import FusedAdamW
    from painter_b200.train_utils import param_groups_lrd
    gold = load_golden("ref_checkpoint.pt")
    scaler = _scaler()
    # save_model stores loss_scaler.state_dict(): empty where the scaler is disabled (no GPU, as when the golden file
    # was made), the scale and growth settings where it is enabled
    want = dict(gold["checkpoint"], scaler=scaler.state_dict())
    # ---- the reference's checkpoint-4.pth, rebuilt: same weights, AdamW over its groups after one step ----
    ref = _ours()
    ref.load_state_dict(synth_state_dict(CFG, 3), strict=True)
    opt_ref = _reference_layout(gold, ref)
    for p in ref.parameters():                      # one AdamW step so that the optimizer has state to carry
        p.grad = torch.full_like(p, 1e-3)
    opt_ref.step()
    tmp_path.mkdir(exist_ok=True)
    path = tmp_path / "checkpoint-4.pth"
    torch.save({"model": ref.state_dict(), "optimizer": opt_ref.state_dict(), "epoch": gold["epoch"],
                "scaler": scaler.state_dict(), "args": _args(tmp_path)}, path)
    assert describe_checkpoint(_load(path)) == want, "rebuilt file differs from the reference's checkpoint"
    # ---- resume into painter_b200 + FusedAdamW ----
    ours = _ours()
    opt = FusedAdamW(param_groups_lrd(ours, 0.05, ours.no_weight_decay(), 0.8), lr=1e-3)
    a = _args(tmp_path)
    assert checkpoint.auto_load_model(a, ours, ours, opt, scaler)
    assert a.resume.endswith("checkpoint-4.pth") and a.start_epoch == 5
    assert _equal_sd(ours.state_dict(), ref.state_dict())
    assert len(opt.param_groups) == len(opt_ref.param_groups)
    for go, gr in zip(opt.param_groups, opt_ref.param_groups):
        assert go["lr_scale"] == gr["lr_scale"] and go["weight_decay"] == gr["weight_decay"]
        for po_, pr in zip(go["params"], gr["params"]):
            assert torch.equal(opt.state[po_]["exp_avg"], opt_ref.state[pr]["exp_avg"])
            assert torch.equal(opt.state[po_]["exp_avg_sq"], opt_ref.state[pr]["exp_avg_sq"])
            assert int(opt.state[po_]["step"]) == int(opt_ref.state[pr]["step"]) == 1
    # ---- write from painter_b200: the same file the reference writes, and it resumes the reference's layout ----
    out2 = tmp_path / "b200"
    checkpoint.save_model(_args(out2), gold["epoch"], ours, ours, opt, scaler)
    mine = _load(out2 / "checkpoint-4.pth")
    assert describe_checkpoint(mine) == want
    # what misc.auto_load_model does with it (misc.py:349-362): strict model load, optimizer load, epoch + 1
    ref2 = _ours()
    opt2 = _reference_layout(gold, ref2)
    ref2.load_state_dict(mine["model"])
    opt2.load_state_dict(mine["optimizer"])
    assert mine["epoch"] + 1 == 5 and _equal_sd(ref2.state_dict(), ours.state_dict())
    p0 = opt2.param_groups[0]["params"][0]
    assert torch.equal(opt2.state[p0]["exp_avg"], opt.state[opt.param_groups[0]["params"][0]]["exp_avg"])


def test_finetune_key_filtering_matches_main_train(tmp_path):
    """main_train.py:199-224 on an MAE-style checkpoint: decoder_embed.* / mask_token of other shapes are dropped,
    extra keys are reported as unexpected, everything else loads.  The reference module's keys and shapes are those
    of its checkpoint in ref_checkpoint.pt."""
    from painter_b200 import checkpoint
    ref_shapes = {k: v[1] for k, v in load_golden("ref_checkpoint.pt")["checkpoint"]["model"].items()}
    sd = synth_state_dict(CFG, 5)
    mae = dict(sd)
    mae["decoder_embed.weight"] = torch.randn(32, 64)           # MAE: Linear(embed_dim, decoder_dim)
    mae["decoder_embed.bias"] = torch.randn(32)
    mae["mask_token"] = torch.randn(1, 1, 32)
    mae["cls_token"] = torch.randn(1, 1, 64)
    del mae["segment_token_x"]
    path = tmp_path / "mae.pth"
    torch.save({"model": mae}, path)
    ours = _ours()
    before = {k: v.clone() for k, v in ours.state_dict().items()}
    assert {k: tuple(v.shape) for k, v in before.items()} == ref_shapes
    msg = checkpoint.load_pretrained(ours, str(path), verbose=False)
    # the reference's inline code, on a module with the reference's keys and shapes
    ck = torch.load(path, map_location="cpu")["model"]
    for k in ["decoder_embed.weight", "decoder_embed.bias", "mask_token"]:
        if k in ck and tuple(ck[k].shape) != ref_shapes[k]:
            del ck[k]
    assert all(tuple(v.shape) == ref_shapes[k] for k, v in ck.items() if k in ref_shapes)   # strict=False loads them
    missing = [k for k in ref_shapes if k not in ck]
    unexpected = [k for k in ck if k not in ref_shapes]
    assert sorted(msg.missing_keys) == sorted(missing)
    assert sorted(msg.unexpected_keys) == sorted(unexpected) == ["cls_token"]
    assert _equal_sd(ours.state_dict(), {k: ck.get(k, before[k]) for k in ref_shapes})
    assert torch.equal(ours.state_dict()["mask_token"], before["mask_token"])       # kept its init: shape mismatch
