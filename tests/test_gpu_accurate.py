"""GPU parity of the fp32-ACCURATE mode (north star: 1e-5 in fp32; SURVEY.md section 8c "fp32 mode": loss rel <= 1e-5,
logits max|d| / max|ref| <= 1e-5) against golden vectors of the unmodified reference (CPU fp32) and against the
unmodified reference executed on a B200 in strict fp32 (TF32 off), stored by oracle/make_golden_gpu.py."""
import pytest
import torch

from oracle import painter_oracle as po
from oracle.synth import synth_inputs

from _common import absmax_rel, build_model, load_golden, norm_rel, rel_max, sampled_max_rel
from _refmods import max_rel, run_module

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _to(dev, *ts):
    return [t.to(dev) for t in ts]


def test_split_gemm_matches_fp64_matmul():
    """The building block: one pk_gemm_bf16 over [l|m|h|m|h|h] x [h|m|l|h|m|h] operands == fp32 GEMM to ~1e-6."""
    from painter_b200 import accurate
    from painter_b200.ops import EPI_F32
    g = torch.Generator().manual_seed(0)
    for M, N, K in ((300, 192, 256), (1568, 1024, 1024), (1568, 3072, 4096)):
        a = torch.randn(M, K, generator=g).cuda()
        b = (torch.randn(N, K, generator=g) * 0.05).cuda()
        bias = torch.randn(N, generator=g).cuda()
        out = accurate._gemm(accurate.split3(a), accurate.split3(b, side_b=True), kind=EPI_F32, bias=bias)
        want = (a.double() @ b.double().t() + bias.double())
        e32 = max_rel(a @ b.t() + bias, want) if True else 0.0
        e = max_rel(out, want)
        print(M, N, K, "split", e, "torch fp32 (may use TF32)", e32)
        assert e < 1e-5, (M, N, K, e)     # fp32 accumulation over K' = 6K terms; measured 1e-6 .. 5e-6


def test_painter_tiny_golden_fp32_mode():
    gold = load_golden("painter_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"], precision="fp32")
    model.eval()
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, **gold["inputs"]))
    with torch.no_grad():
        loss, pred, _ = model(imgs, tgts, mask, valid)
    ev = gold["eval"]
    assert abs(loss.item() - ev["loss"].item()) <= TOL * abs(ev["loss"].item()), (loss.item(), ev["loss"].item())
    assert rel_max(pred, ev["pred"]) <= TOL, rel_max(pred, ev["pred"])
    it = gold["interp"]          # 64x32 input on the 128x64 model: interpolated abs-pos / rel-pos tables
    i2, t2, mk2, v2 = _to("cuda", *synth_inputs(cfg, **it["inputs"]))
    with torch.no_grad():
        loss, pred, _ = model(i2, t2, mk2, v2)
    assert abs(loss.item() - it["loss"].item()) <= TOL * abs(it["loss"].item())
    assert rel_max(pred, it["pred"]) <= TOL, rel_max(pred, it["pred"])


def test_seggpt_tiny_golden_fp32_mode_auto_selected():
    """precision = "auto": called outside autocast under no_grad (as seggpt_engine.run_one_image does) the module
    computes in the fp32-accurate mode; prompts 1/2/3 incl. the feature ensemble and both seg types."""
    gold = load_golden("seggpt_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"], precision="auto")
    model.eval()
    h, w = cfg.grid
    for c in gold["cases"]:
        x, t, _, _ = synth_inputs(cfg, c["P"], c["seed"])
        bm = torch.zeros(1, h * w)
        bm[:, h * w // 2:] = 1
        seg = torch.full((c["P"], 1), float(c["seg_type"]))
        with torch.no_grad():
            loss, pred, _ = model(x.cuda(), t.cuda(), bm.cuda(), torch.ones_like(t).cuda(), seg.cuda(),
                                  c["merge_between_batch"])
        assert abs(loss.item() - c["loss"].item()) <= TOL * abs(c["loss"].item()), c["P"]
        assert rel_max(pred, c["pred"]) <= TOL, (c["P"], rel_max(pred, c["pred"]))
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):     # auto -> bf16 under autocast
            _, pred_b, _ = model(x.cuda(), t.cuda(), bm.cuda(), torch.ones_like(t).cuda(), seg.cuda(),
                                 c["merge_between_batch"])
        assert 1e-4 < rel_max(pred_b, c["pred"]) < 4e-2


def test_seggpt_vitl_run_one_image_fp32_mode_vs_reference_fp32():
    """configs[2] at full size through run_one_image (painter_b200.seggpt_engine, bit-identical to the unmodified
    seggpt_engine.run_one_image): the module in its default "auto" precision against the reference module in strict
    fp32 on a B200 (tests/golden/ref_seggpt_vitl.pt, oracle/make_golden_gpu.py), over a seeded sample of 65536 of the
    602112 result values."""
    from painter_b200 import seggpt_engine
    gold = load_golden("ref_seggpt_vitl.pt")
    cfg = po.PainterConfig(seggpt=True)
    dev = torch.device("cuda")
    model, _ = build_model(cfg, 3, precision="auto")
    model.eval()
    rep = {}
    for c in gold["cases"]:
        P, seg = c["P"], c["seg_type"]
        x, t, _, _ = synth_inputs(cfg, P, 40 + P)
        img = x.permute(0, 2, 3, 1).double().numpy()
        tgt = t.permute(0, 2, 3, 1).double().numpy()
        model.seg_type = seg
        out_o = seggpt_engine.run_one_image(img, tgt, model, dev)
        mr = sampled_max_rel(out_o, c["out_fp32"])
        err = mr * c["out_fp32"]["absmax"] / 255.0
        rep[f"P{P}_{seg}"] = {"max_abs_err_over_255": err, "max_rel": mr}
        assert err <= TOL, rep
        assert norm_rel(out_o, c["out_fp32"]) <= TOL and absmax_rel(out_o, c["out_fp32"]) <= TOL, rep
    print(rep)


def test_painter_vitl_fp32_mode_vs_reference_fp32():
    """The stock ViT-L Painter in fp32 mode against the reference in strict fp32 on a B200
    (tests/golden/ref_vitl_896x448_fwd.pt): loss, and the logits over a seeded sample of 131072 of 1.2 M values."""
    ref = load_golden("ref_vitl_896x448_fwd.pt")
    cfg = po.PainterConfig()
    args = [t.cuda() for t in synth_inputs(cfg, 1, 21, valid_kind="mixed")]
    model, _ = build_model(cfg, 1, precision="fp32")
    model.eval()
    with torch.no_grad():
        loss_o, pred_o, _ = run_module(model, args, backward=False)
    le = abs(loss_o.item() - ref["loss_fp32"]) / abs(ref["loss_fp32"])
    pe = sampled_max_rel(pred_o, ref["pred_fp32"])
    print("fp32 mode: loss rel", le, "logits max-rel", pe)
    assert le <= TOL and pe <= TOL, (le, pe)
    assert norm_rel(pred_o, ref["pred_fp32"]) <= TOL and absmax_rel(pred_o, ref["pred_fp32"]) <= TOL
