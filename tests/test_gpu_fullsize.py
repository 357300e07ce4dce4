"""GPU parity at the BENCHMARKED shapes against the UNMODIFIED reference, following the SURVEY.md section 8(c) protocol:

  * loss: |ours - ref| <= 1e-3 |ref| against the reference in fp32 (TF32 off) AND under torch.autocast('cuda', bf16);
  * logits / gradients: err(ours, fp32 reference) <= 1.5 x err(reference-bf16-autocast, fp32 reference), per
    tensor (RMS-rel) and globally.  With $PAINTER_PARITY_REPORT set, the measured ratios are written to that JSON file
    (committed copy of a B200 run: profiles/r02_parity.json).

The reference side was executed on a B200 by oracle/make_golden_gpu.py and is stored under tests/golden/ref_*.pt:
losses, the reference's own bf16 error computed on the full tensors, and seeded samples of its fp32 logits and
gradients (the RMS of ours - reference is estimated on the sample; tensors up to the sample size are stored whole).

Covers BASELINE.json configs[1] (ViT-L 896x448, B=1 eval and B=8 train with the module's own CUDA DropPath draws),
configs[2] (SegGPT ViT-L through run_one_image, 1 and 2 prompts), configs[4] (1792x896, N=6272: full forward + one
Block forward/backward) and the unmodified engine_train.train_one_epoch loop.
"""
import gc
import json
import os
import types

import numpy as np
import pytest
import torch

from oracle import painter_oracle as po
from oracle.synth import synth_inputs

from _common import absmax_rel, build_model, load_golden, norm_rel, sampled_max_rel, sampled_rms_rel, sampled_sq_err
from _refmods import build_reference, have_reference, rms_rel, run_module, strict_fp32

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-3          # north star: loss within 1e-3 relative of the reference
NOISE_RATIO = 1.5        # SURVEY 8(c): ours <= 1.5 x the reference's own bf16 error


def _record(name, payload):
    path = os.environ.get("PAINTER_PARITY_REPORT")
    if not path:
        return
    try:
        with open(path) as f:
            allr = json.load(f)
    except (OSError, ValueError):
        allr = {}
    allr[name] = payload
    with open(path, "w") as f:
        json.dump(allr, f, indent=1, sort_keys=True)


def _free():
    gc.collect()
    torch.cuda.empty_cache()


def _cuda(*ts):
    return [t.cuda() for t in ts]


def _check_against_noise(tag, loss_o, loss_f, loss_b, lo, lb, rows, glob, extra=None):
    """rows: (name, err ours, err reference-bf16, numel) per gradient tensor; glob: global RMS-rel of both."""
    glob = dict(glob, ratio=glob["ours"] / max(glob["ref_bf16"], 1e-30))
    ratios = [(r[0], r[1], r[2], r[1] / max(r[2], 1e-30), r[3]) for r in rows]
    worst = sorted(ratios, key=lambda r: -r[3])[:12]
    rep = {
        "loss": {"ours": loss_o, "ref_fp32": loss_f, "ref_bf16": loss_b,
                 "rel_vs_fp32": abs(loss_o - loss_f) / abs(loss_f), "rel_vs_bf16": abs(loss_o - loss_b) / abs(loss_b),
                 "ref_bf16_rel_vs_fp32": abs(loss_b - loss_f) / abs(loss_f)},
        "logits_rms_rel": {"ours": lo, "ref_bf16": lb, "ratio": lo / lb},
        "grads_global_rms_rel": glob,
        "grads_tensors": len(ratios),
        "grads_tensors_over_1p5": sum(1 for r in ratios if r[3] > NOISE_RATIO),
        "grads_worst_ratio": [{"name": r[0], "ours": r[1], "ref_bf16": r[2], "ratio": r[3], "numel": r[4]}
                              for r in worst],
        "grads_median_ratio": float(np.median([r[3] for r in ratios])),
    }
    if extra:
        rep.update(extra)
    _record(tag, rep)
    print(tag, json.dumps({k: rep[k] for k in ("loss", "logits_rms_rel", "grads_global_rms_rel",
                                                "grads_tensors_over_1p5", "grads_median_ratio")}))
    assert rep["loss"]["rel_vs_fp32"] <= LOSS_TOL and rep["loss"]["rel_vs_bf16"] <= LOSS_TOL, rep["loss"]
    assert lo <= NOISE_RATIO * lb, rep["logits_rms_rel"]
    assert glob["ratio"] <= NOISE_RATIO, glob
    bad = [(r[0], r[1], r[2]) for r in ratios if r[3] > NOISE_RATIO]
    assert not bad, bad[:10]


def _sampled_grad_rows(g_o, stored):
    """Per-tensor rows and the global RMS-rel of ours against the stored reference gradient samples; also asserts
    that each whole tensor's norm is within the same noise rule of the reference's."""
    rows, se, sf, bad = [], 0.0, 0.0, []
    for k, c, eb in zip(stored["names"], stored["fp32"], stored["ref_bf16_rms_rel"]):
        rows.append((k, sampled_rms_rel(g_o[k], c), eb, c["numel"]))
        if norm_rel(g_o[k], c) > NOISE_RATIO * eb:
            bad.append((k, norm_rel(g_o[k], c), eb))
        se += sampled_sq_err(g_o[k], c)
        sf += c["sumsq"]
    assert not bad, ("whole-tensor gradient norms", bad[:10])
    return rows, {"ours": (se / sf) ** 0.5, "ref_bf16": stored["ref_bf16_global_rms_rel"]}


def test_vitl_b1_eval_fwd_bwd_all_grads_vs_reference():
    """configs[1] geometry, B=1, eval: every gradient tensor (370.7 M values) against the reference in fp32 and in bf16
    autocast - the error on a seeded sample of up to 320 values per tensor, the norm over the whole tensor."""
    ref, ref_g = load_golden("ref_vitl_896x448_fwd.pt"), load_golden("ref_vitl_896x448_grads.pt")
    cfg = po.PainterConfig()
    args = _cuda(*synth_inputs(cfg, 1, 21, valid_kind="mixed"))
    model, _ = build_model(cfg, 1)
    loss_o, pred_o, g_o = run_module(model, args)
    del model
    _free()
    assert set(ref_g["names"]) <= set(g_o)
    rows, glob = _sampled_grad_rows(g_o, ref_g)
    lo = sampled_rms_rel(pred_o, ref["pred_fp32"])
    assert norm_rel(pred_o, ref["pred_fp32"]) <= NOISE_RATIO * ref["pred_ref_bf16_rms_rel"]
    assert absmax_rel(pred_o, ref["pred_fp32"]) <= NOISE_RATIO * ref["pred_ref_bf16_max_rel"]
    _check_against_noise("vitl_896x448_b1_eval", loss_o.item(), ref["loss_fp32"], ref["loss_ref_bf16"], lo,
                         ref["pred_ref_bf16_rms_rel"], rows, glob,
                         extra={"logits_max_rel": {"ours": sampled_max_rel(pred_o, ref["pred_fp32"]),
                                                   "ref_bf16": ref["pred_ref_bf16_max_rel"]}})


def test_vitl_b8_train_step_vs_reference_same_cuda_rng():
    """configs[1]: B=8 TRAIN mode under torch.autocast(bf16) - the bench's GEMM plans (M = 25088 / 12544) and the
    module's own CUDA DropPath draws (same seed => the reference draws the same masks, timm DropPath order/dtype).
    The fp32 truth is the pinned oracle restatement replaying the recorded masks; the stored reference side is its
    bf16 loss and its bf16 error against that truth."""
    ref = load_golden("ref_vitl_b8_train.pt")
    cfg = po.PainterConfig()
    B, seed = 8, 1234
    args = _cuda(*synth_inputs(cfg, B, 5, valid_kind="mixed"))
    # --- ours, recording the DropPath scales the module drew on the device ---
    model, sd = build_model(cfg, 2)
    drawn = {}
    orig = model._drop_scales

    def rec(i, Bp, dev):
        out = orig(i, Bp, dev)
        drawn[i] = out
        return out

    model._drop_scales = rec
    loss_o, pred_o, g_o = run_module(model, args, train=True, autocast=torch.bfloat16, seed=seed)
    del model
    _free()
    # --- fp32 truth: the (pinned) oracle restatement on CUDA in strict fp32 with the recorded masks ---
    drops = []
    for i in range(cfg.depth):
        Bp = 2 * B if i <= cfg.merge_idx else B
        a, m = drawn[i]
        one = torch.ones(Bp, device="cuda")
        drops.append((one if a is None else a.float(), one if m is None else m.float()))
    sdc = {k: v.cuda().requires_grad_(True) for k, v in sd.items()}
    with strict_fp32():
        loss_f, pred_f, _ = po.forward(sdc, cfg, *args, drops=drops)
        loss_f.backward()
    g_f = {k: v.grad.detach() for k, v in sdc.items()}
    loss_f, pred_f = loss_f.detach(), pred_f.detach()
    n_dropped = int(sum((d[0] == 0).sum().item() + (d[1] == 0).sum().item() for d in drops))
    rows = [(k, rms_rel(g_o[k], g_f[k]), eb, g_f[k].numel()) for k, eb in zip(ref["names"], ref["ref_bf16_rms_rel"])]
    so = sum((g_o[k].double() - g_f[k].double()).pow(2).sum().item() for k in ref["names"])
    sf = sum(g_f[k].double().pow(2).sum().item() for k in ref["names"])
    _check_against_noise("vitl_896x448_b8_train", loss_o.item(), loss_f.item(), ref["loss_ref_bf16"],
                         rms_rel(pred_o, pred_f), ref["pred_ref_bf16_rms_rel"], rows,
                         {"ours": (so / sf) ** 0.5, "ref_bf16": ref["ref_bf16_global_rms_rel"]},
                         extra={"droppath_branches_dropped": n_dropped})
    assert n_dropped > 0, "DropPath never fired: the train-mode path was not exercised"


def test_seggpt_vitl_run_one_image_unmodified_engine():
    """configs[2]: run_one_image (painter_b200.seggpt_engine, bit-identical to the unmodified seggpt_engine.py:26-53 -
    tests/test_gpu_inference.py) on the painter_b200 SegGPT module against the reference module in strict fp32 on
    the same numpy inputs: 1 prompt (no ensemble) and 2 prompts (feature ensemble), both seg types."""
    from painter_b200 import seggpt_engine
    gold = load_golden("ref_seggpt_vitl.pt")
    cfg = po.PainterConfig(seggpt=True)
    dev = torch.device("cuda")
    model, _ = build_model(cfg, 3)
    model.eval()
    rep = {}
    for c in gold["cases"]:
        P, seg = c["P"], c["seg_type"]
        x, t, _, _ = synth_inputs(cfg, P, 40 + P)
        img = x.permute(0, 2, 3, 1).double().numpy()
        tgt = t.permute(0, 2, 3, 1).double().numpy()
        model.seg_type = seg
        out_o = seggpt_engine.run_one_image(img, tgt, model, dev)
        assert tuple(out_o.shape) == tuple(c["shape"]) == (448, 448, 3) and out_o.dtype == torch.float64
        eo, eb = sampled_rms_rel(out_o, c["out_fp32"]), c["ref_bf16_rms_rel"]
        assert norm_rel(out_o, c["out_fp32"]) <= NOISE_RATIO * eb, (P, seg)
        rep[f"P{P}_{seg}"] = {"rms_rel_ours": eo, "rms_rel_ref_bf16": eb, "ratio": eo / eb,
                              "max_abs_ours_of_255": sampled_max_rel(out_o, c["out_fp32"]) * c["out_fp32"]["absmax"],
                              "max_abs_ref_bf16_of_255": c["ref_bf16_max_abs"]}
        assert eo <= NOISE_RATIO * eb, rep
    _record("seggpt_vitl_run_one_image", rep)
    print(rep)


def test_long_sequence_1792x896_forward_and_block_backward():
    """configs[4]: Painter(img_size=(1792, 896)) - N = 6272 tokens, native 223/111-row tables: full forward B=1 and
    a single Block forward/backward at N = 6272 (SURVEY 8c: the full backward oracle does not fit)."""
    ref = load_golden("ref_long_1792x896.pt")
    cfg = po.PainterConfig(img_size=(1792, 896))
    args = _cuda(*synth_inputs(cfg, 1, 77))
    model, sd = build_model(cfg, 4)
    model.eval()
    with torch.no_grad():
        loss_o, pred_o, _ = run_module(model, args, backward=False)
    loss_o = loss_o.item()
    rep = {"loss_rel_vs_fp32": abs(loss_o - ref["loss_fp32"]) / abs(ref["loss_fp32"]),
           "loss_rel_vs_bf16": abs(loss_o - ref["loss_ref_bf16"]) / abs(ref["loss_ref_bf16"]),
           "logits_rms_rel": {"ours": sampled_rms_rel(pred_o, ref["pred_fp32"]),
                              "ref_bf16": ref["pred_ref_bf16_rms_rel"]}}
    assert rep["loss_rel_vs_fp32"] <= LOSS_TOL and rep["loss_rel_vs_bf16"] <= LOSS_TOL, rep
    assert rep["logits_rms_rel"]["ours"] <= NOISE_RATIO * rep["logits_rms_rel"]["ref_bf16"], rep
    assert norm_rel(pred_o, ref["pred_fp32"]) <= NOISE_RATIO * ref["pred_ref_bf16_rms_rel"]
    # ---- one Block at N = 6272, batch 2 (the x / y halves), forward + backward ----
    from painter_b200.engine import BlockFn
    h, w = cfg.grid
    C = cfg.embed_dim
    blk = model.blocks[7]
    g = torch.Generator().manual_seed(5)
    z0 = torch.randn(2, h, w, C, generator=g).cuda()
    dz = torch.randn(2, h, w, C, generator=g).cuda()
    for p in model.parameters():
        p.grad = None
    zin = z0.reshape(2 * h * w, C).clone().requires_grad_(True)
    prm = blk.params()
    out_o = BlockFn.apply(zin, None, None, *prm, (2, h, w, cfg.num_heads, 1e-6, 0, 0, 0))
    out_o.backward(dz.reshape(2 * h * w, C))
    g_o = {"blocks.7." + n: p.grad.detach().float().clone() for n, p in blk.named_parameters()}
    g_o["dx"] = zin.grad.detach().reshape(2, h, w, C)
    rows, glob = _sampled_grad_rows(g_o, ref["block_grads"])
    assert norm_rel(out_o, ref["block_out_fp32"]) <= NOISE_RATIO * ref["block_out_ref_bf16_rms_rel"]
    glob["ratio"] = glob["ours"] / glob["ref_bf16"]
    rep["block_out_rms_rel"] = {"ours": sampled_rms_rel(out_o, ref["block_out_fp32"]),
                                "ref_bf16": ref["block_out_ref_bf16_rms_rel"]}
    rep["block_grads_global"] = glob
    rep["block_grads"] = [{"name": r[0], "ours": r[1], "ref_bf16": r[2], "ratio": r[1] / r[2]} for r in rows]
    _record("long_1792x896", rep)
    print(json.dumps(rep["block_grads_global"]), rep["block_out_rms_rel"])
    assert rep["block_out_rms_rel"]["ours"] <= NOISE_RATIO * rep["block_out_rms_rel"]["ref_bf16"], rep
    assert glob["ratio"] <= NOISE_RATIO, glob
    bad = [(r[0], r[1], r[2]) for r in rows if r[1] > NOISE_RATIO * r[2]]
    assert not bad, bad


def test_stock_weights_on_double_resolution_input_interpolated_tables():
    """SURVEY 8(d) config 5 variant: the stock 896x448 model fed a 1792x896 canvas (rel-pos tables linearly resized
    111 -> 223 / 55 -> 111 rows, abs-pos bicubic 14x14 -> 112x56; vitdet_utils.py:75-86,141-153)."""
    ref = load_golden("ref_stock_1792x896_input.pt")
    cfg = po.PainterConfig()
    args = _cuda(*synth_inputs(cfg, 1, 78, size=(1792, 896)))
    model, _ = build_model(cfg, 5)
    model.eval()
    with torch.no_grad():
        loss_o, pred_o, _ = run_module(model, args, backward=False)
    rep = {"loss_rel_vs_fp32": abs(loss_o.item() - ref["loss_fp32"]) / abs(ref["loss_fp32"]),
           "logits_rms_rel": {"ours": sampled_rms_rel(pred_o, ref["pred_fp32"]),
                              "ref_bf16": ref["pred_ref_bf16_rms_rel"]}}
    _record("stock_weights_1792x896_input", rep)
    assert norm_rel(pred_o, ref["pred_fp32"]) <= NOISE_RATIO * ref["pred_ref_bf16_rms_rel"]
    assert rep["loss_rel_vs_fp32"] <= LOSS_TOL, rep
    assert rep["logits_rms_rel"]["ours"] <= NOISE_RATIO * rep["logits_rms_rel"]["ref_bf16"], rep


def _train_args():
    return types.SimpleNamespace(accum_iter=1, clip_grad=3.0, lr=1e-4, min_lr=0.0, warmup_epochs=0, epochs=15,
                                 log_wandb=False)


@pytest.mark.skipif(not have_reference(), reason="drives the unmodified reference training loop: needs the reference "
                                                  "tree (PAINTER_REFERENCE or oracle/_ref)")
def test_unmodified_train_one_epoch_drives_the_module():
    """engine_train.train_one_epoch (UNMODIFIED, engine_train.py:34-144: fp16 autocast context, loss.item(),
    NativeScalerWithGradNormCount -> GradScaler / clip_grad_norm_ / AdamW, torch.cuda.synchronize, MetricLogger) runs
    against the painter_b200 module exactly as against the reference module, on the same loader and RNG seeds."""
    from oracle import ref_loader
    et, misc = ref_loader.engine_train(), ref_loader.misc()
    lrd = ref_loader.lr_decay()
    cfg = po.PainterConfig()
    dev = torch.device("cuda")
    loader = [tuple(t.pin_memory() for t in synth_inputs(cfg, 2, 90 + i)) for i in range(2)]

    def drive(m):
        groups = lrd.param_groups_lrd(m, 0.05, no_weight_decay_list=m.no_weight_decay(), layer_decay=0.8)
        opt = torch.optim.AdamW(groups, lr=1e-4, betas=(0.9, 0.999))
        scaler = misc.NativeScalerWithGradNormCount()
        out = []
        for epoch in range(2):
            torch.manual_seed(700 + epoch)
            stats = et.train_one_epoch(m, loader[epoch:epoch + 1], opt, dev, epoch, scaler, log_writer=None,
                                       global_rank=0, args=_train_args())
            out.append(stats)
        return out

    ref = build_reference(cfg, 6, stock_factory=True)
    s_ref = drive(ref)
    del ref
    _free()
    model, _ = build_model(cfg, 6)
    s_our = drive(model)
    rep = {"ref": s_ref, "ours": s_our}
    _record("train_one_epoch_unmodified", rep)
    print(rep)
    for a, b in zip(s_our, s_ref):
        assert np.isfinite(a["loss"]) and np.isfinite(a["grad_norm"])
    # iteration 0: same weights, same batch, same DropPath draws -> same loss and gradient norm
    assert abs(s_our[0]["loss"] - s_ref[0]["loss"]) <= LOSS_TOL * abs(s_ref[0]["loss"]), rep
    if np.isfinite(s_ref[0]["grad_norm"]):   # the reference's fp16 backward may overflow at the initial loss scale
        assert abs(s_our[0]["grad_norm"] - s_ref[0]["grad_norm"]) <= 2e-2 * abs(s_ref[0]["grad_norm"]), rep
    # iteration 1 runs on the AdamW-updated weights (first Adam step ~ lr * sign(g): amplifies rounding differences)
    assert abs(s_our[1]["loss"] - s_ref[1]["loss"]) <= 1e-2 * abs(s_ref[1]["loss"]), rep
