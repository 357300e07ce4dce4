"""TEST INFRASTRUCTURE - golden data for the full-size GPU parity tests, by EXECUTING THE UNMODIFIED REFERENCE on a GPU.

    PAINTER_REFERENCE=<reference checkout> python -m oracle.make_golden_gpu [OUT_DIR]    # default: tests/golden

Stores the reference side of tests/test_gpu_fullsize.py and tests/test_gpu_accurate.py: losses, the reference's own
bf16-autocast error against its fp32 result (per tensor, computed on the full tensors), and seeded samples of the fp32
outputs and gradients (oracle.synth.compact) so that every file stays well under 1 MB.  Weights and inputs are
regenerated from their seeds by oracle/synth.py, exactly as the tests do.
"""
import gc
import os
import sys

import torch

from . import ref_loader
from .painter_oracle import PainterConfig
from .synth import compact, synth_inputs, synth_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from _refmods import build_reference, max_rel, rms_rel, run_module, strict_fp32  # noqa: E402

GRAD_SAMPLES = 320          # per gradient tensor (exact below that size)
PRED_SAMPLES = 131072       # logits of one 896x448 image: 1.2 M values
OUT_SAMPLES = 65536         # one SegGPT result image: 448 x 448 x 3 values


def _free():
    gc.collect()
    torch.cuda.empty_cache()


def _cuda(*ts):
    return [t.cuda() for t in ts]


def _grads(g_f, g_b):
    names = list(g_f)
    return {"names": names,
            "fp32": [compact(g_f[k], GRAD_SAMPLES, i) for i, k in enumerate(names)],
            "ref_bf16_rms_rel": [rms_rel(g_b[k], g_f[k]) for k in names],
            "ref_bf16_global_rms_rel": (sum((g_b[k].double() - g_f[k].double()).pow(2).sum().item() for k in names) /
                                        sum(g_f[k].double().pow(2).sum().item() for k in names)) ** 0.5}


def vitl_896x448(out):
    """tests/test_gpu_fullsize.py::test_vitl_b1_eval_fwd_bwd_all_grads_vs_reference and
    tests/test_gpu_accurate.py::test_painter_vitl_fp32_mode_vs_reference_fp32: stock factory, weight seed 1, B = 1,
    input seed 21 with mixed valid maps, eval mode."""
    cfg = PainterConfig()
    args = _cuda(*synth_inputs(cfg, 1, 21, valid_kind="mixed"))
    ref = build_reference(cfg, 1, stock_factory=True)
    with strict_fp32():
        loss_f, pred_f, g_f = run_module(ref, args)
    loss_b, pred_b, g_b = run_module(ref, args, autocast=torch.bfloat16)
    del ref
    _free()
    torch.save({"loss_fp32": loss_f.item(), "loss_ref_bf16": loss_b.item(), "pred_fp32": compact(pred_f, PRED_SAMPLES),
                "pred_ref_bf16_rms_rel": rms_rel(pred_b, pred_f), "pred_ref_bf16_max_rel": max_rel(pred_b, pred_f)},
               os.path.join(out, "ref_vitl_896x448_fwd.pt"))
    torch.save(_grads(g_f, g_b), os.path.join(out, "ref_vitl_896x448_grads.pt"))
    print("vitl 896x448 loss", loss_f.item(), loss_b.item())


def vitl_b8_train(out):
    """tests/test_gpu_fullsize.py::test_vitl_b8_train_step_vs_reference_same_cuda_rng: the reference's bf16 train step
    (its DropPath masks drawn from CUDA seed 1234) against the fp32 oracle replaying the masks painter_b200 drew from
    the same seed."""
    from oracle import painter_oracle as po
    from _common import build_model
    cfg = PainterConfig()
    B, seed = 8, 1234
    args = _cuda(*synth_inputs(cfg, B, 5, valid_kind="mixed"))
    model, sd = build_model(cfg, 2)
    drawn = {}
    orig = model._drop_scales

    def rec(i, Bp, dev):
        drawn[i] = orig(i, Bp, dev)
        return drawn[i]

    model._drop_scales = rec
    run_module(model, args, train=True, autocast=torch.bfloat16, seed=seed)
    del model
    _free()
    ref = build_reference(cfg, 2, stock_factory=True)
    loss_b, pred_b, g_b = run_module(ref, args, train=True, autocast=torch.bfloat16, seed=seed)
    del ref
    _free()
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
    g = _grads(g_f, g_b)
    torch.save({"loss_ref_bf16": loss_b.item(), "pred_ref_bf16_rms_rel": rms_rel(pred_b, pred_f.detach()),
                "names": g["names"], "ref_bf16_rms_rel": g["ref_bf16_rms_rel"],
                "ref_bf16_global_rms_rel": g["ref_bf16_global_rms_rel"]},
               os.path.join(out, "ref_vitl_b8_train.pt"))
    print("vitl b8 train loss", loss_b.item(), loss_f.item())


def seggpt_vitl(out):
    """tests/test_gpu_fullsize.py::test_seggpt_vitl_run_one_image_unmodified_engine and
    tests/test_gpu_accurate.py::test_seggpt_vitl_run_one_image_fp32_mode_vs_reference_fp32: the unmodified
    seggpt_engine.run_one_image on the reference module (weight seed 3) in strict fp32, 1 prompt (instance) and
    2 prompts (semantic), inputs seeded 40 + P; plus the reference module's own bf16-autocast error."""
    se = ref_loader.seggpt_engine()
    cfg = PainterConfig(seggpt=True)
    dev = torch.device("cuda")
    ref = build_reference(cfg, 3, stock_factory=True).eval()
    cases = []
    for P, seg in ((1, "instance"), (2, "semantic")):
        x, t, _, _ = synth_inputs(cfg, P, 40 + P)
        img = x.permute(0, 2, 3, 1).double().numpy()
        tgt = t.permute(0, 2, 3, 1).double().numpy()
        ref.seg_type = seg
        with strict_fp32():
            out_f = se.run_one_image(img, tgt, ref, dev)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            bm = torch.zeros(1, ref.patch_embed.num_patches)
            bm[:, ref.patch_embed.num_patches // 2:] = 1
            xt, tt = torch.tensor(img).permute(0, 3, 1, 2), torch.tensor(tgt).permute(0, 3, 1, 2)
            sgt = torch.ones(P, 1) if seg == "instance" else torch.zeros(P, 1)
            _, yb, _ = ref(xt.float().to(dev), tt.float().to(dev), bm.to(dev), torch.ones_like(tt).float().to(dev),
                           sgt.to(dev), 0 if P > 1 else -1)
        yb = ref.unpatchify(yb.float()).permute(0, 2, 3, 1).cpu()
        out_b = torch.clip((yb[0, yb.shape[1] // 2:] * se.imagenet_std + se.imagenet_mean) * 255, 0, 255)
        cases.append({"P": P, "seg_type": seg, "shape": tuple(out_f.shape), "out_fp32": compact(out_f, OUT_SAMPLES),
                      "ref_bf16_rms_rel": rms_rel(out_b, out_f),
                      "ref_bf16_max_abs": (out_b - out_f).abs().max().item()})
    torch.save({"cases": cases}, os.path.join(out, "ref_seggpt_vitl.pt"))
    print("seggpt", [(c["P"], c["ref_bf16_rms_rel"]) for c in cases])


def long_1792x896(out):
    """tests/test_gpu_fullsize.py::test_long_sequence_1792x896_forward_and_block_backward: Painter(img_size=(1792,
    896)) with weight seed 4, input seed 77, eval forward; then blocks.7 alone at N = 6272 forward + backward on seeded
    inputs (torch.Generator seed 5)."""
    cfg = PainterConfig(img_size=(1792, 896))
    args = _cuda(*synth_inputs(cfg, 1, 77))
    ref = build_reference(cfg, 4).eval()
    with torch.no_grad():
        with strict_fp32():
            loss_f, pred_f, _ = run_module(ref, args, backward=False)
        loss_b, pred_b, _ = run_module(ref, args, autocast=torch.bfloat16, backward=False)
    del ref
    _free()
    h, w = cfg.grid
    C = cfg.embed_dim
    g = torch.Generator().manual_seed(5)
    z0 = torch.randn(2, h, w, C, generator=g).cuda()
    dz = torch.randn(2, h, w, C, generator=g).cuda()
    sd = synth_state_dict(cfg, 4)
    mp = ref_loader.models_painter()
    rb = mp.Block(dim=C, num_heads=cfg.num_heads, mlp_ratio=4, qkv_bias=True, drop_path=0.0,
                  norm_layer=lambda d: torch.nn.LayerNorm(d, eps=1e-6), use_rel_pos=True, window_size=0,
                  input_size=(h, w)).cuda()
    rb.load_state_dict({k[len("blocks.7."):]: v for k, v in sd.items() if k.startswith("blocks.7.")}, strict=True)

    def ref_block(autocast):
        for p in rb.parameters():
            p.grad = None
        zin = z0.clone().requires_grad_(True)
        if autocast:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                o = rb(zin)
        else:
            with strict_fp32():
                o = rb(zin)
        o.float().backward(dz)
        gr = {"blocks.7." + n: p.grad.detach().float().clone() for n, p in rb.named_parameters()}
        gr["dx"] = zin.grad.detach().clone()
        return o.detach().float(), gr

    out_f, g_f = ref_block(False)
    out_b, g_b = ref_block(True)
    grads = _grads(g_f, g_b)
    grads["fp32"] = [compact(g_f[k], 4096, i) for i, k in enumerate(grads["names"])]
    torch.save({"loss_fp32": loss_f.item(), "loss_ref_bf16": loss_b.item(), "pred_fp32": compact(pred_f, 65536),
                "pred_ref_bf16_rms_rel": rms_rel(pred_b, pred_f),
                "block_out_fp32": compact(out_f, 65536), "block_out_ref_bf16_rms_rel": rms_rel(out_b, out_f),
                "block_grads": grads},
               os.path.join(out, "ref_long_1792x896.pt"))
    print("long loss", loss_f.item(), loss_b.item())


def stock_1792x896_input(out):
    """tests/test_gpu_fullsize.py::test_stock_weights_on_double_resolution_input_interpolated_tables: the stock
    896x448 model (weight seed 5) fed a 1792x896 canvas (input seed 78), eval forward."""
    cfg = PainterConfig()
    args = _cuda(*synth_inputs(cfg, 1, 78, size=(1792, 896)))
    ref = build_reference(cfg, 5, stock_factory=True).eval()
    with torch.no_grad():
        with strict_fp32():
            loss_f, pred_f, _ = run_module(ref, args, backward=False)
        loss_b, pred_b, _ = run_module(ref, args, autocast=torch.bfloat16, backward=False)
    del ref
    _free()
    torch.save({"loss_fp32": loss_f.item(), "pred_fp32": compact(pred_f, 65536),
                "pred_ref_bf16_rms_rel": rms_rel(pred_b, pred_f)},
               os.path.join(out, "ref_stock_1792x896_input.pt"))
    print("stock 1792x896 input loss", loss_f.item())


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(out, exist_ok=True)
    assert ref_loader.available(), "reference tree not found (set PAINTER_REFERENCE or stage it into oracle/_ref)"
    for fn in (vitl_896x448, vitl_b8_train, seggpt_vitl, long_1792x896, stock_1792x896_input):
        fn(out)
        _free()
    for f in sorted(os.listdir(out)):
        print(f, os.path.getsize(os.path.join(out, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
