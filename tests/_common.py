"""Helpers shared by the GPU parity tests."""
import os

import torch

from oracle import painter_oracle as po
from oracle.synth import sample_positions, synth_inputs, synth_state_dict

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def build_model(cfg: po.PainterConfig, seed, device="cuda", precision="bf16"):
    """painter_b200 module of the same geometry as `cfg`, loaded with the synthetic reference-format weights.
    precision: the module's arithmetic mode, pinned to "bf16" unless a test is about the fp32-accurate / auto modes."""
    from functools import partial
    from painter_b200 import models_painter, models_seggpt
    cls = models_seggpt.SegGPT if cfg.seggpt else models_painter.Painter
    m = cls(img_size=tuple(cfg.img_size), patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
            num_heads=cfg.num_heads, drop_path_rate=cfg.drop_path_rate, window_size=cfg.window_size, qkv_bias=True,
            mlp_ratio=cfg.mlp_ratio, norm_layer=partial(torch.nn.LayerNorm, eps=cfg.ln_eps),
            window_block_indexes=list(cfg.window_block_indexes), residual_block_indexes=[], use_rel_pos=True,
            out_feature="last_feat", decoder_embed_dim=cfg.decoder_embed_dim, loss_func=cfg.loss_func,
            pretrain_img_size=cfg.pretrain_img_size)
    sd = synth_state_dict(cfg, seed)
    m.load_state_dict(sd, strict=True)
    m.precision = precision
    return m.to(device), sd


def rel_max(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def rel_rms(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-12)).item()


def _at_sample(a, c):
    """`a` at the positions of the stored reference sample `c` (oracle.synth.compact), and the sampled values."""
    pos = sample_positions(c["numel"], c["n"], c["seed"])
    a = torch.as_tensor(a).detach().reshape(-1)
    assert a.numel() == c["numel"], (a.numel(), c["numel"])
    return a[pos.to(a.device)].double().cpu(), c["val"].double()


def sampled_sq_err(a, c):
    """sum((a - ref)^2) over the whole tensor, estimated from the stored sample (exact when it holds every value)."""
    x, r = _at_sample(a, c)
    return (x - r).pow(2).mean().item() * c["numel"]


def sampled_rms_rel(a, c):
    """rms(a - ref) / rms(ref) with rms(ref) exact and rms(a - ref) from the stored sample."""
    return (sampled_sq_err(a, c) / max(c["sumsq"], 1e-300)) ** 0.5


def norm_rel(a, c):
    """| ||a|| - ||ref|| | / ||ref|| over the WHOLE tensor, from the stored exact sum of squares of the reference.
    Bounded by rms(a - ref) / rms(ref), so every RMS-rel tolerance applies to it; it sees the values the sample misses."""
    n = torch.as_tensor(a).detach().double().pow(2).sum().sqrt().item()
    r = max(c["sumsq"], 1e-300) ** 0.5
    return abs(n - r) / r


def absmax_rel(a, c):
    """| max|a| - max|ref| | / max|ref| over the WHOLE tensor; bounded by the max-rel error of a against ref."""
    m = torch.as_tensor(a).detach().abs().max().item()
    return abs(m - c["absmax"]) / max(c["absmax"], 1e-300)


def sampled_max_rel(a, c):
    """max |a - ref| over the stored sample / max |ref| over the whole tensor."""
    x, r = _at_sample(a, c)
    return ((x - r).abs().max() / max(c["absmax"], 1e-300)).item()
