"""TEST INFRASTRUCTURE — deterministic synthetic weights and inputs shared by the golden generator, the
parity tests, smoke() and bench.py.  Weights are drawn from a seeded CPU generator (same torch build here
and on the GPU box => bit-identical), so fixtures only need to store OUTPUTS of the reference."""
import torch

from .painter_oracle import PainterConfig


def param_shapes(cfg: PainterConfig):
    """Reference state-dict keys and shapes (SURVEY.md §8 a1; models_painter.py:263-333)."""
    C, p, dd = cfg.embed_dim, cfg.patch_size, cfg.decoder_embed_dim
    h, w = cfg.grid
    d = C // cfg.num_heads
    hid = int(C * cfg.mlp_ratio)
    npos = (cfg.pretrain_img_size // p) ** 2 + 1
    out = {"mask_token": (1, 1, 1, C), "segment_token_x": (1, 1, 1, C), "segment_token_y": (1, 1, 1, C)}
    if cfg.seggpt:
        out["type_token_cls"] = (1, 1, 1, C)
        out["type_token_ins"] = (1, 1, 1, C)
    out["pos_embed"] = (1, npos, C)
    out["patch_embed.proj.weight"] = (C, 3, p, p)
    out["patch_embed.proj.bias"] = (C,)
    for i in range(cfg.depth):
        ws = cfg.window_size if i in tuple(cfg.window_block_indexes) else 0
        rh, rw = (2 * ws - 1, 2 * ws - 1) if ws > 0 else (2 * h - 1, 2 * w - 1)
        b = f"blocks.{i}."
        out[b + "norm1.weight"] = (C,)
        out[b + "norm1.bias"] = (C,)
        out[b + "attn.rel_pos_h"] = (rh, d)
        out[b + "attn.rel_pos_w"] = (rw, d)
        out[b + "attn.qkv.weight"] = (3 * C, C)
        out[b + "attn.qkv.bias"] = (3 * C,)
        out[b + "attn.proj.weight"] = (C, C)
        out[b + "attn.proj.bias"] = (C,)
        out[b + "norm2.weight"] = (C,)
        out[b + "norm2.bias"] = (C,)
        out[b + "mlp.fc1.weight"] = (hid, C)
        out[b + "mlp.fc1.bias"] = (hid,)
        out[b + "mlp.fc2.weight"] = (C, hid)
        out[b + "mlp.fc2.bias"] = (C,)
    out["norm.weight"] = (C,)
    out["norm.bias"] = (C,)
    out["decoder_embed.weight"] = (p * p * dd, 4 * C)
    out["decoder_embed.bias"] = (p * p * dd,)
    out["decoder_pred.0.weight"] = (dd, dd, 3, 3)
    out["decoder_pred.0.bias"] = (dd,)
    out["decoder_pred.1.weight"] = (dd,)
    out["decoder_pred.1.bias"] = (dd,)
    out["decoder_pred.3.weight"] = (3, dd, 1, 1)
    out["decoder_pred.3.bias"] = (3,)
    return out


def synth_state_dict(cfg: PainterConfig, seed=0, dtype=torch.float32):
    """All parameters live (rel_pos randomised, biases non-zero, LN gains around 1)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shp in param_shapes(cfg).items():
        t = torch.randn(shp, generator=g)
        if k.endswith("norm1.weight") or k.endswith("norm2.weight") or k in ("norm.weight", "decoder_pred.1.weight"):
            t = 1 + 0.1 * t
        elif k.endswith(".bias"):
            t = 0.05 * t
        elif "rel_pos" in k:
            t = 0.1 * t
        elif k.startswith("decoder_pred") and k.endswith("weight"):
            t = t * (1.0 / (shp[1] * shp[2] * shp[3]) ** 0.5)
        elif k in ("patch_embed.proj.weight",):
            t = 0.02 * t
        elif k.endswith(".weight"):
            t = t * min(0.02 * (1024 / shp[1]) ** 0.5, 0.08)
        else:  # tokens, pos_embed
            t = 0.02 * t
        sd[k] = t.to(dtype)
    return sd


def synth_inputs(cfg: PainterConfig, B, seed, mask_kind="random", valid_kind="ones", dark_sample=None,
                 size=None):
    g = torch.Generator().manual_seed(seed)
    H, W = size or cfg.img_size
    h, w = H // cfg.patch_size, W // cfg.patch_size
    imgs = torch.randn(B, 3, H, W, generator=g)
    tgts = torch.randn(B, 3, H, W, generator=g)
    if mask_kind == "half":
        mask = torch.zeros(B, h, w, dtype=torch.int32)
        mask[:, h // 2:] = 1
    else:
        mask = (torch.rand(B, h, w, generator=g) < 0.5).to(torch.int32)
    valid = torch.ones(B, 3, H, W)
    if valid_kind == "mixed":
        r = torch.rand(B, 3, H, W, generator=g)
        valid[r < 0.1] = 0.0
        valid[r > 0.95] = 10.0
    if dark_sample is not None:  # triggers inds_ign (models_painter.py:446-448)
        std = torch.tensor([0.229, 0.224, 0.225])[:, None, None]
        mean = torch.tensor([0.485, 0.456, 0.406])[:, None, None]
        tgts[dark_sample] = (torch.zeros(3, H, W) - mean) / std
    return imgs, tgts, mask, valid


def compact(t, n=4096, seed=0):
    """A reference tensor too large to store whole: its size, exact sum of squares and max |x|, and its values at n
    positions drawn (with replacement) from a generator seeded by `seed`; sample_positions() regenerates them."""
    t = t.detach().float().cpu().reshape(-1)
    idx = sample_positions(t.numel(), n, seed)
    return {"numel": t.numel(), "n": n, "seed": seed, "val": t[idx].clone(),
            "sumsq": float(t.double().pow(2).sum()), "absmax": float(t.abs().max())}


def sample_positions(numel, n, seed):
    if numel <= n:
        return torch.arange(numel)
    return torch.randint(numel, (n,), generator=torch.Generator().manual_seed(seed))


def fingerprint(sd):
    """Cheap checksum guarding against RNG drift between torch builds."""
    s = 0.0
    for k in sorted(sd):
        s += float(sd[k].double().abs().sum())
    return s
