"""TEST INFRASTRUCTURE — generate golden vectors by EXECUTING THE UNMODIFIED REFERENCE.

Run with the reference tree available (PAINTER_REFERENCE or oracle/_ref):   python -m oracle.make_golden
Writes small fixtures to tests/golden/*.pt: {cfg, state_dict, inputs, outputs(loss, pred, grads...)}.
Small model geometries are used so that every fixture file stays under 1 MB; the reference classes are the real
`models_painter.Painter` / `models_seggpt.SegGPT` constructed with non-stock sizes (depth must stay 24:
the taps [5,11,17,23] are hard-coded, models_painter.py:416).
"""
import os
import random
from functools import partial

import numpy as np
import torch

from . import ref_loader
from .painter_oracle import PainterConfig
from .synth import compact, fingerprint, synth_inputs, synth_state_dict

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def build_ref(cfg: PainterConfig, seed=0):
    torch.manual_seed(seed)
    mod = ref_loader.models_seggpt() if cfg.seggpt else ref_loader.models_painter()
    cls = mod.SegGPT if cfg.seggpt else mod.Painter
    m = cls(img_size=tuple(cfg.img_size), patch_size=cfg.patch_size, embed_dim=cfg.embed_dim,
            depth=cfg.depth, num_heads=cfg.num_heads, drop_path_rate=cfg.drop_path_rate,
            window_size=cfg.window_size, qkv_bias=True, mlp_ratio=cfg.mlp_ratio,
            norm_layer=partial(torch.nn.LayerNorm, eps=cfg.ln_eps),
            window_block_indexes=list(cfg.window_block_indexes), residual_block_indexes=[],
            use_rel_pos=True, out_feature="last_feat", decoder_embed_dim=cfg.decoder_embed_dim,
            loss_func=cfg.loss_func, pretrain_img_size=cfg.pretrain_img_size)
    # all-live deterministic weights (rel_pos tables are zero-initialised in the reference,
    # models_painter.py:66-67, which would leave the bias path untested)
    missing = m.load_state_dict(synth_state_dict(cfg, seed), strict=True)
    return m


def run_ref_painter(m, cfg, imgs, tgts, mask, valid, train):
    m.train(train)
    for p in m.parameters():
        p.grad = None
    rng_state = torch.get_rng_state()
    loss, pred, bmask = m(imgs.clone(), tgts.clone(), mask.clone(), valid.clone())
    loss.backward()
    grads = {n: p.grad.clone() for n, p in m.named_parameters()}
    return dict(loss=loss.detach(), pred=pred.detach(), mask=bmask, grads=grads, rng_state=rng_state)


TINY = dict(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64, window_size=2)
GRAD_KEYS = ["mask_token", "pos_embed", "patch_embed.proj.weight", "patch_embed.proj.bias",
             "segment_token_x", "segment_token_y", "blocks.0.attn.rel_pos_h", "blocks.0.attn.rel_pos_w",
             "blocks.1.attn.qkv.weight", "blocks.1.attn.qkv.bias", "blocks.2.attn.proj.weight",
             "blocks.2.mlp.fc2.bias", "blocks.3.norm1.weight", "blocks.3.norm1.bias",
             "blocks.7.mlp.fc1.weight", "blocks.23.attn.rel_pos_w", "blocks.23.mlp.fc2.weight",
             "norm.weight", "norm.bias", "decoder_embed.bias", "decoder_pred.0.weight",
             "decoder_pred.0.bias", "decoder_pred.1.weight", "decoder_pred.1.bias",
             "decoder_pred.3.weight", "decoder_pred.3.bias"]


def _slim(r, keys, whole=None):
    """Gradient norms of every tensor; the gradients of `keys`, stored whole up to `whole` values and as a seeded
    sample of `whole` values (oracle.synth.compact) above that, so that each fixture file stays under 1 MB."""
    r["grad_norms"] = {n: g.norm().item() for n, g in r["grads"].items()}
    r["grads"] = {n: r["grads"][n] for n in keys if n in r["grads"] and r["grads"][n].numel() <= 70000}
    if whole is not None:
        r["grads"] = {n: compact(g, whole, i) if g.numel() > whole else g for i, (n, g) in enumerate(r["grads"].items())}
    r.pop("rng_state", None)
    return r


LOSS_GRAD_KEYS = ["decoder_pred.3.weight", "decoder_pred.3.bias", "decoder_pred.1.weight", "decoder_pred.0.bias",
                  "blocks.23.mlp.fc2.bias", "mask_token"]


def make_losses():
    """The reference's other `loss_func` values (models_painter.py:453-458: l1, l2, l1l2) on the tiny geometry,
    eval mode, mixed valid + one dark sample; written to painter_tiny_losses.pt (python -m oracle.make_golden losses)."""
    out = dict(cases=[])
    for lf in ("l1", "l2", "l1l2"):
        cfg = PainterConfig(**TINY, loss_func=lf)
        m = build_ref(cfg, 2)
        inp = dict(B=2, seed=21, mask_kind="random", valid_kind="mixed", dark_sample=0)
        imgs, tgts, mask, valid = synth_inputs(cfg, **inp)
        ev = _slim(run_ref_painter(m, cfg, imgs, tgts, mask, valid, train=False), LOSS_GRAD_KEYS)
        out["cases"].append(dict(cfg=cfg.__dict__, weight_seed=2, inputs=inp, loss=ev["loss"], grads=ev["grads"],
                                 grad_norms={k: ev["grad_norms"][k] for k in LOSS_GRAD_KEYS}))
        print("loss_func", lf, "loss", ev["loss"].item())
    torch.save(out, os.path.join(GOLD, "painter_tiny_losses.pt"))


def make_vitl():
    """The stock factory painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1() at the benchmark geometry,
    torch-CPU fp32, eval forward, B = 1, weight seed 3, input seed 11: loss, mask, a seeded sample of the logits, and
    the window size every block was built with; written to ref_vitl_cpu_fwd.pt (python -m oracle.make_golden vitl)."""
    cfg = PainterConfig()
    sd = synth_state_dict(cfg, 3)
    imgs, tgts, mask, valid = synth_inputs(cfg, 1, 11)
    model = ref_loader.models_painter().painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1()
    model.load_state_dict(sd, strict=True)
    model.eval()
    with torch.no_grad():
        loss, pred, bmask = model(imgs, tgts, bool_masked_pos=mask, valid=valid.clone())
    torch.save(dict(loss=loss.item(), pred=compact(pred, 131072), mask=bmask,
                    window_sizes=[b.window_size for b in model.blocks]),
               os.path.join(GOLD, "ref_vitl_cpu_fwd.pt"))
    print("vitl cpu loss", loss.item())


DATAPATH_TYPES = ["nyuv2_image2depth", "ade20k_image2semantic", "coco_image2panoptic_sem_seg", "coco_image2pose",
                  "coco_image2panoptic_inst", "ssid_image2denoise"]


def datapath_pairs(root, H=64, W=64):
    """Writes the 12 image / target PNG pairs and pairs.json that tests/test_gpu_datapath.py feeds PairDataset."""
    import json
    from PIL import Image
    rng = np.random.RandomState(0)
    pairs = []
    for t in DATAPATH_TYPES:
        for k in range(2):
            img = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
            tgt = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
            tgt[: H // 2, : W // 3] = 0                       # black region -> below every threshold
            if "pose" in t and k == 0:
                tgt[:] = 0                                    # nearly no foreground -> valid = 0 branch
                tgt[0, 0] = 200
            if "inst" in t and k == 1:
                tgt[:] = 0
            ip, tp = f"{t}_{k}_img.png", f"{t}_{k}_tgt.png"
            Image.fromarray(img).save(os.path.join(root, ip))
            Image.fromarray(tgt).save(os.path.join(root, tp))
            pairs.append({"image_path": ip, "target_path": tp, "type": t})
    jp = os.path.join(root, "pairs.json")
    with open(jp, "w") as f:
        json.dump(pairs, f)
    return pairs, jp


def to_normalised(u8):
    """[3, H, W] uint8 -> ImageNet-normalised float32, the transform the data-path test hands PairDataset."""
    mean = torch.tensor([0.485, 0.456, 0.406])[:, None, None]
    std = torch.tensor([0.229, 0.224, 0.225])[:, None, None]
    return (u8.float() / 255.0 - mean) / std


def make_datapath():
    """Reference side of tests/test_gpu_datapath.py, written to ref_datapath.pt (python -m oracle.make_golden
    datapath): statistics of 1024 MaskingGenerator draws (main_train.py:256-260, random / numpy seed 0), and the
    targets (as the uint8 pixels they were normalised from) and `valid` maps PairDataset.__getitem__ returns for the
    pairs of datapath_pairs() (random / torch seed 1), plus one _combine_images call."""
    import tempfile
    MG = ref_loader.masking_generator().MaskingGenerator
    h, w, target, n = 56, 28, 784, 1024
    ref = MG((h, w), num_masking_patches=target, max_num_patches=392, min_num_patches=16)
    random.seed(0)
    np.random.seed(0)
    mr = np.stack([ref() for _ in range(n)]).astype(np.float64)
    assert (mr.reshape(n, -1).sum(1) == target).all()
    blockiness = ((mr[:, 1:, :] == mr[:, :-1, :]).mean() + (mr[:, :, 1:] == mr[:, :, :-1]).mean()) / 2
    out = dict(masks=dict(blockiness=float(blockiness), mean_map=torch.from_numpy(mr.mean(0)),
                          row_marginal=torch.from_numpy(mr.mean((0, 2))), col_marginal=torch.from_numpy(mr.mean((0, 1)))))
    PD = ref_loader.pairdataset()

    def tf(img, tgt, i1, i2):
        f = lambda im: to_normalised(torch.from_numpy(np.array(im)).permute(2, 0, 1))
        return f(img), f(tgt)

    with tempfile.TemporaryDirectory() as d:
        pairs, jp = datapath_pairs(d)
        ds = PD.PairDataset(d, [jp], transform=tf, masked_position_generator=MG((8, 4), 16, 4),
                            use_two_pairs=True, half_mask_ratio=0.0)
        random.seed(1)
        torch.manual_seed(1)
        tg, vd = [], []
        for i in range(len(ds)):
            _, tgt, _, valid = ds[i]
            mean = torch.tensor([0.485, 0.456, 0.406])[:, None, None]
            std = torch.tensor([0.229, 0.224, 0.225])[:, None, None]
            u8 = ((tgt * std + mean) * 255.0).round().clamp(0, 255).to(torch.uint8)
            assert torch.equal(to_normalised(u8), tgt)          # the stored pixels reproduce the target bit for bit
            tg.append(u8)
            vd.append(valid)
        g = torch.Generator().manual_seed(0)
        a, b = torch.randn(2, 3, 8, 4, generator=g), torch.randn(2, 3, 8, 4, generator=g)
        out.update(types=[p["type"] for p in pairs], targets_u8=torch.stack(tg), valid=torch.stack(vd).to(torch.int8),
                   combine=dict(a=a, b=b, out=ds._combine_images(a[0], b[0])))
    assert set(torch.stack(vd).unique().tolist()) == {0.0, 1.0, 10.0}
    torch.save(out, os.path.join(GOLD, "ref_datapath.pt"))
    print("datapath blockiness", blockiness)


CKPT_CFG = dict(img_size=(64, 32), embed_dim=64, num_heads=1, decoder_embed_dim=64)


def describe_checkpoint(ckpt):
    """Everything in a checkpoint-<epoch>.pth except tensor data, which is replaced by (shape, dtype, sha256 of the
    bytes): equal descriptions mean equal files for every loader.  args.output_dir (a run's own path) is left out."""
    import hashlib

    def d(v):
        if torch.is_tensor(v):
            t = v.detach().cpu().contiguous()
            return ("tensor", tuple(t.shape), str(t.dtype),
                    hashlib.sha256(t.reshape(-1).view(torch.uint8).numpy().tobytes()).hexdigest())
        if isinstance(v, dict):
            return {k: d(x) for k, x in v.items()}
        if isinstance(v, (list, tuple)):
            return [d(x) for x in v]
        return v

    out = {k: d(v) for k, v in ckpt.items() if k != "args"}
    out["keys"] = list(ckpt.keys())
    if "args" in ckpt:
        out["args"] = {k: v for k, v in vars(ckpt["args"]).items() if k != "output_dir"}
        out["args_type"] = type(ckpt["args"]).__name__
    return out


def make_checkpoint():
    """Reference side of tests/test_checkpoint.py, written to ref_checkpoint.pt (python -m oracle.make_golden
    checkpoint): the unmodified misc.save_model's checkpoint of a Painter (64x32, embed 64, weight seed 3) with
    torch.optim.AdamW over the unmodified lr_decay.param_groups_lrd groups (wd 0.05, layer decay 0.8, lr 1e-3) after
    one step on gradients of 1e-3, as describe_checkpoint() sees it, and the parameter names of every group."""
    import tempfile
    import types
    misc, lrd = ref_loader.misc(), ref_loader.lr_decay()
    mp = ref_loader.models_painter()
    ref = mp.Painter(img_size=(64, 32), patch_size=16, embed_dim=64, depth=24, num_heads=1, drop_path_rate=0.1,
                     window_size=2, qkv_bias=True, mlp_ratio=4, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6),
                     window_block_indexes=[], residual_block_indexes=[], use_rel_pos=True, decoder_embed_dim=64)
    ref.load_state_dict(synth_state_dict(PainterConfig(**CKPT_CFG), 3), strict=True)
    groups = lrd.param_groups_lrd(ref, 0.05, ref.no_weight_decay(), 0.8)
    opt = torch.optim.AdamW(groups, lr=1e-3)
    for p in ref.parameters():
        p.grad = torch.full_like(p, 1e-3)
    opt.step()
    names = {id(p): n for n, p in ref.named_parameters()}
    with tempfile.TemporaryDirectory() as d:
        args = types.SimpleNamespace(output_dir=d, resume="", auto_resume=True, start_epoch=0)
        misc.save_model(args, 4, ref, ref, opt, misc.NativeScalerWithGradNormCount())
        ckpt = torch.load(os.path.join(d, "checkpoint-4.pth"), map_location="cpu", weights_only=False)
    torch.save(dict(checkpoint=describe_checkpoint(ckpt), epoch=4,
                    group_names=[[names[id(p)] for p in g["params"]] for g in opt.param_groups]),
               os.path.join(GOLD, "ref_checkpoint.pt"))
    print("checkpoint", len(ckpt["model"]), "tensors,", len(opt.param_groups), "groups")


def main():
    import sys
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    if "losses" in sys.argv[1:]:
        make_losses()
        return
    if "vitl" in sys.argv[1:]:
        make_vitl()
        return
    if "datapath" in sys.argv[1:]:
        make_datapath()
        return
    if "checkpoint" in sys.argv[1:]:
        make_checkpoint()
        return
    make_losses()
    make_vitl()
    make_datapath()
    make_checkpoint()
    # Fixtures store SEEDS (weights/inputs are regenerated by oracle/synth.py) + reference OUTPUTS.
    # ---- 1. Painter tiny, eval + train (DropPath drawn from torch.manual_seed(77)), random mask,
    #         mixed valid, one dark sample (inds_ign path)
    cfg = PainterConfig(**TINY)
    m = build_ref(cfg, 0)
    inp = dict(B=3, seed=11, mask_kind="random", valid_kind="mixed", dark_sample=1)
    imgs, tgts, mask, valid = synth_inputs(cfg, **inp)
    ev = _slim(run_ref_painter(m, cfg, imgs, tgts, mask, valid, train=False), GRAD_KEYS, 16384)
    torch.manual_seed(77)
    tr = _slim(run_ref_painter(m, cfg, imgs, tgts, mask, valid, train=True), GRAD_KEYS, 16384)
    # 64x32 input on the 128x64 model: rel-pos / abs-pos interpolation path (vitdet_utils.py:75-86,141-153)
    i2, t2, mk2, v2 = synth_inputs(cfg, 2, 9, size=(64, 32))
    m.eval()
    l2, p2, _ = m(i2, t2, mk2, v2)
    torch.save(dict(cfg=cfg.__dict__, weight_seed=0, weight_fp=fingerprint(synth_state_dict(cfg, 0)),
                    inputs=inp, eval=ev, train_seed=77,
                    interp=dict(inputs=dict(B=2, seed=9, size=(64, 32)), loss=l2.detach(), pred=p2.detach())),
               os.path.join(GOLD, "painter_tiny.pt"))
    torch.save(tr, os.path.join(GOLD, "painter_tiny_train.pt"))
    print("painter_tiny eval loss", ev["loss"].item(), "train loss", tr["loss"].item(), "interp", l2.item())

    # ---- 2. Painter tiny with REAL window blocks (parameterised, non-stock feature; ws=7 pads 8x4 -> 14x7)
    cfgw = PainterConfig(**{**TINY, "window_size": 7}, window_block_indexes=(0, 1, 3, 4, 6, 7))
    mw = build_ref(cfgw, 3)
    inpw = dict(B=2, seed=5)
    iw, tw, mkw, vw = synth_inputs(cfgw, **inpw)
    evw = _slim(run_ref_painter(mw, cfgw, iw, tw, mkw, vw, train=False),
                ["blocks.0.attn.rel_pos_h", "blocks.2.attn.rel_pos_h", "blocks.1.attn.qkv.weight", "pos_embed"])
    torch.save(dict(cfg=cfgw.__dict__, weight_seed=3, inputs=inpw, eval=evw),
               os.path.join(GOLD, "painter_tiny_window.pt"))
    print("window eval loss", evw["loss"].item())

    # ---- 3. SegGPT tiny: P=1/3/2 prompts, both seg types, half mask (as seggpt_engine.run_one_image)
    cfgs = PainterConfig(**TINY, seggpt=True)
    ms = build_ref(cfgs, 5).eval()
    out = dict(cfg=cfgs.__dict__, weight_seed=5, cases=[])
    h, w = cfgs.grid
    for P, st in ((1, 0), (3, 1), (2, 0)):
        x, t, _, _ = synth_inputs(cfgs, P, 100 + P)
        bm = torch.zeros(1, h * w)
        bm[:, h * w // 2:] = 1
        seg = torch.full((P, 1), float(st))
        fe = 0 if P > 1 else -1
        with torch.no_grad():
            loss, y, mk = ms(x, t, bm, torch.ones_like(t), seg, fe)
        out["cases"].append(dict(P=P, seed=100 + P, seg_type=st, merge_between_batch=fe, loss=loss, pred=y))
        print("seggpt P", P, "loss", loss.item())
    torch.save(out, os.path.join(GOLD, "seggpt_tiny.pt"))

    # ---- 4. BEiT block masks from the reference MaskingGenerator (main_train.py:256-260), full geometry
    mg = ref_loader.masking_generator().MaskingGenerator
    random.seed(3)
    np.random.seed(3)
    gen = mg((56, 28), num_masking_patches=784, max_num_patches=392, min_num_patches=16)
    masks = np.stack([gen() for _ in range(16)]).astype(np.uint8)
    torch.save(torch.from_numpy(np.packbits(masks, axis=-1)), os.path.join(GOLD, "beit_masks_56x28.pt"))
    print("masks", masks.shape, masks.sum((1, 2))[:4])
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
