"""TEST INFRASTRUCTURE: the UNMODIFIED reference modules (oracle/ref_loader.py: $PAINTER_REFERENCE or the
staged byte-for-byte copy oracle/_ref) loaded with the same synthetic weights as the painter_b200 module.
"""
from contextlib import contextmanager
from functools import partial

import torch

from oracle import painter_oracle as po
from oracle import ref_loader
from oracle.synth import synth_state_dict


def have_reference():
    return ref_loader.available()


def build_reference(cfg: po.PainterConfig, seed, device="cuda", stock_factory=False):
    """Reference `Painter` / `SegGPT` with the geometry of cfg; stock_factory=True calls the zero-argument factory
    (painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1 / seggpt_vit_large_patch16_input896x448)."""
    mod = ref_loader.models_seggpt() if cfg.seggpt else ref_loader.models_painter()
    if stock_factory:
        fn = (mod.seggpt_vit_large_patch16_input896x448 if cfg.seggpt else
              mod.painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1)
        m = fn()
    else:
        cls = mod.SegGPT if cfg.seggpt else mod.Painter
        m = cls(img_size=tuple(cfg.img_size), patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
                num_heads=cfg.num_heads, drop_path_rate=cfg.drop_path_rate, window_size=cfg.window_size,
                qkv_bias=True, mlp_ratio=cfg.mlp_ratio, norm_layer=partial(torch.nn.LayerNorm, eps=cfg.ln_eps),
                window_block_indexes=list(cfg.window_block_indexes), residual_block_indexes=[], use_rel_pos=True,
                out_feature="last_feat", decoder_embed_dim=cfg.decoder_embed_dim, loss_func=cfg.loss_func,
                pretrain_img_size=cfg.pretrain_img_size)
    m.load_state_dict(synth_state_dict(cfg, seed), strict=True)
    return m.to(device)


@contextmanager
def strict_fp32():
    """fp32 reference arithmetic on CUDA: no TF32 in matmul or cuDNN (SURVEY.md section 8c)."""
    a, b = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    prec = torch.get_float32_matmul_precision()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = a
        torch.backends.cudnn.allow_tf32 = b
        torch.set_float32_matmul_precision(prec)


def run_module(m, args, train=False, autocast=None, seed=None, backward=True, **kw):
    """One forward(+backward) of a reference or painter_b200 module; returns (loss, pred, {name: grad})."""
    m.train(train)
    for p in m.parameters():
        p.grad = None
    if seed is not None:
        torch.manual_seed(seed)
    imgs, tgts, mask, valid = [t.clone() for t in args]
    if autocast is None:
        loss, pred, _ = m(imgs, tgts, mask, valid, **kw)
    else:
        with torch.autocast("cuda", dtype=autocast):
            loss, pred, _ = m(imgs, tgts, mask, valid, **kw)
    grads = None
    if backward:
        loss.float().backward()
        grads = {n: p.grad.detach().float().clone() for n, p in m.named_parameters()}
        for p in m.parameters():
            p.grad = None
    return loss.detach().float(), pred.detach().float(), grads


def rms_rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-30)).item()


def max_rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def grad_report(g_ours, g_refbf16, g_fp32):
    """Per-tensor and global RMS-rel errors of `ours` and of the reference's own bf16-autocast run against fp32."""
    rows = []
    so = sb = sf = 0.0
    for k, gf in g_fp32.items():
        eo, eb = rms_rel(g_ours[k], gf), rms_rel(g_refbf16[k], gf)
        rows.append((k, eo, eb, eo / max(eb, 1e-30), gf.numel()))
        so += (g_ours[k].double() - gf.double()).pow(2).sum().item()
        sb += (g_refbf16[k].double() - gf.double()).pow(2).sum().item()
        sf += gf.double().pow(2).sum().item()
    glob = dict(ours=(so / sf) ** 0.5, ref_bf16=(sb / sf) ** 0.5)
    glob["ratio"] = glob["ours"] / max(glob["ref_bf16"], 1e-30)
    return rows, glob
