"""Pins the CPU oracle (oracle/painter_oracle.py) against golden vectors produced by executing the
unmodified reference (oracle/make_golden.py), at the toy geometries and at the benchmark geometry.  CPU only."""
import os

import torch

from oracle import painter_oracle as po
from oracle.synth import fingerprint, synth_inputs, synth_state_dict

from conftest import GOLDEN
from _common import sampled_max_rel


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def _rel(a, b):
    """max |a - b| / max |b|; b may be a stored seeded sample of the reference tensor (oracle.synth.compact)."""
    if isinstance(b, dict):
        return sampled_max_rel(a, b)
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def _oracle_run(cfg, sd, imgs, tgts, mask, valid, drops=None, grads=True, **kw):
    sd = {k: v.clone().requires_grad_(grads) for k, v in sd.items()}
    loss, pred, m = po.forward(sd, cfg, imgs, tgts, mask, valid, drops=drops, **kw)
    g = {}
    if grads:
        loss.backward()
        g = {k: v.grad for k, v in sd.items()}
    return loss.detach(), pred.detach(), m, g


def test_painter_tiny_eval_and_train():
    gold = _load("painter_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    sd = synth_state_dict(cfg, gold["weight_seed"])
    assert abs(fingerprint(sd) - gold["weight_fp"]) < 1e-6 * gold["weight_fp"], "synthetic weight RNG drift"
    imgs, tgts, mask, valid = synth_inputs(cfg, **gold["inputs"])
    loss, pred, m, g = _oracle_run(cfg, sd, imgs, tgts, mask, valid)
    ev = gold["eval"]
    assert abs(loss.item() - ev["loss"].item()) < 2e-6 * abs(ev["loss"].item())
    assert _rel(pred, ev["pred"]) < 2e-5
    assert torch.equal(m, ev["mask"])
    for k, ref in ev["grads"].items():
        assert _rel(g[k], ref) < 2e-4, k
    for k, n in ev["grad_norms"].items():
        assert abs(g[k].norm().item() - n) <= 2e-4 * max(n, 1e-6), k
    # train mode: replay the reference's DropPath draws
    torch.manual_seed(gold["train_seed"])
    drops = po.draw_drop_scales(cfg, imgs.shape[0])
    loss, pred, _, g = _oracle_run(cfg, sd, imgs, tgts, mask, valid, drops=drops)
    tr = _load("painter_tiny_train.pt")
    assert abs(loss.item() - tr["loss"].item()) < 2e-6 * abs(tr["loss"].item())
    assert _rel(pred, tr["pred"]) < 2e-5
    for k, ref in tr["grads"].items():
        assert _rel(g[k], ref) < 2e-4, k
    # interpolation path: 64x32 input on the 128x64 model
    it = gold["interp"]
    i2, t2, mk2, v2 = synth_inputs(cfg, **it["inputs"])
    loss, pred, _, _ = _oracle_run(cfg, sd, i2, t2, mk2, v2, grads=False)
    assert abs(loss.item() - it["loss"].item()) < 2e-6
    assert _rel(pred, it["pred"]) < 2e-5


def test_painter_tiny_other_loss_functions():
    """models_painter.py:453-458: loss_func in {l1, l2, l1l2} (smoothl1 is the stock one, covered above)."""
    gold = _load("painter_tiny_losses.pt")
    assert [c["cfg"]["loss_func"] for c in gold["cases"]] == ["l1", "l2", "l1l2"]
    for c in gold["cases"]:
        cfg = po.PainterConfig(**c["cfg"])
        sd = synth_state_dict(cfg, c["weight_seed"])
        imgs, tgts, mask, valid = synth_inputs(cfg, **c["inputs"])
        loss, _, _, g = _oracle_run(cfg, sd, imgs, tgts, mask, valid)
        assert abs(loss.item() - c["loss"].item()) < 2e-6 * abs(c["loss"].item()), cfg.loss_func
        for k, ref in c["grads"].items():
            assert _rel(g[k], ref) < 2e-4, (cfg.loss_func, k)
        for k, n in c["grad_norms"].items():
            assert abs(g[k].norm().item() - n) <= 2e-4 * max(n, 1e-6), (cfg.loss_func, k)


def test_painter_tiny_window():
    gold = _load("painter_tiny_window.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    sd = synth_state_dict(cfg, gold["weight_seed"])
    imgs, tgts, mask, valid = synth_inputs(cfg, **gold["inputs"])
    loss, pred, _, g = _oracle_run(cfg, sd, imgs, tgts, mask, valid)
    ev = gold["eval"]
    assert abs(loss.item() - ev["loss"].item()) < 2e-6
    assert _rel(pred, ev["pred"]) < 2e-5
    for k, ref in ev["grads"].items():
        assert _rel(g[k], ref) < 2e-4, k


def test_seggpt_tiny():
    gold = _load("seggpt_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    sd = synth_state_dict(cfg, gold["weight_seed"])
    h, w = cfg.grid
    for c in gold["cases"]:
        x, t, _, _ = synth_inputs(cfg, c["P"], c["seed"])
        bm = torch.zeros(1, h * w)
        bm[:, h * w // 2:] = 1
        seg = torch.full((c["P"], 1), float(c["seg_type"]))
        loss, pred, _, _ = _oracle_run(cfg, sd, x, t, bm, torch.ones_like(t), grads=False, seg_type=seg,
                                       merge_between_batch=c["merge_between_batch"])
        assert abs(loss.item() - c["loss"].item()) < 2e-6, c["P"]
        assert _rel(pred, c["pred"]) < 2e-5, c["P"]


def test_patchify_roundtrip():
    x = torch.randn(2, 3, 64, 32)
    assert torch.equal(po.unpatchify(po.patchify(x, 16), 16), x)


def test_live_reference_stock_constructor_is_all_global():
    """SURVEY.md §0.1: the reference's stock factory builds 24 global-attention blocks (tuple-of-lists bug); the
    window size of every block it built is stored in ref_vitl_cpu_fwd.pt, and painter_b200's factory agrees."""
    from painter_b200 import models_painter
    gold = _load("ref_vitl_cpu_fwd.pt")
    assert gold["window_sizes"] == [0] * 24
    assert [b.window_size for b in models_painter.painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1().blocks] \
        == gold["window_sizes"]


def test_live_reference_full_size_forward_pins_the_oracle_at_the_benchmark_geometry():
    """The oracle against the UNMODIFIED reference module at the geometry the benchmark runs (ViT-L, 896x448, the stock
    factory) - not only at the toy geometry of the golden vectors: eval-mode forward, B = 1, same seeded weights and
    inputs, torch-CPU fp32 on both sides (reference side stored by `python -m oracle.make_golden vitl`).  Loss within
    1e-6 relative, logits within 1e-5 of their range over a seeded sample of 131072 of the 1.2 M values."""
    torch.set_num_threads(min(32, torch.get_num_threads()))
    gold = _load("ref_vitl_cpu_fwd.pt")
    cfg = po.PainterConfig()
    sd = synth_state_dict(cfg, 3)
    imgs, tgts, mask, valid = synth_inputs(cfg, 1, 11)
    with torch.no_grad():
        ol, op, om = po.forward(sd, cfg, imgs, tgts, mask, valid)
    assert abs(ol.item() - gold["loss"]) <= 1e-6 * abs(gold["loss"]), (ol.item(), gold["loss"])
    assert _rel(op, gold["pred"]) <= 1e-5, _rel(op, gold["pred"])
    assert torch.equal(om, gold["mask"])
