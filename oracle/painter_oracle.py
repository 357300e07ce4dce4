"""TEST INFRASTRUCTURE — CPU restatement (torch, fp32 or fp64) of the reference hot path.

This file is the parity ORACLE for painter_b200.  It is imported only by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs; the product path
(painter_b200/*) never imports it and has no CPU fallback.

Parity status: PINNED — tests/test_oracle_golden.py checks this restatement against golden vectors
produced by executing the unmodified reference (oracle/make_golden.py), at toy geometries and at the
benchmark geometry.
The reference itself ships no tests or golden vectors (SURVEY.md §4).

It restates, as a pure function of a reference-format state_dict:
  A1 PatchEmbed                      Painter/util/vitdet_utils.py:178-186
  A2 token assembly                  Painter/models_painter.py:392-409 (SegGPT: models_seggpt.py:414-420)
  A3 Block                           Painter/models_painter.py:216-235 (SegGPT merge: models_seggpt.py:220-231)
  A4 Attention + decomposed rel-pos  Painter/models_painter.py:73-89, util/vitdet_utils.py:63-125
  A5 early merge + taps              Painter/models_painter.py:411-418
  A7 decoder                         Painter/models_painter.py:420-431, util/vitdet_utils.py:204-209
  A8 loss / patchify                 Painter/models_painter.py:355-383,433-462 (SegGPT: models_seggpt.py:448-469)
Third-party arithmetic (torch ops; timm==0.3.2 Mlp/DropPath, not vendored in the reference) is restated
from the published definitions: Mlp = fc1 -> erf-GELU -> fc2; DropPath = x/keep * floor(keep + U[0,1)).
Gradients are obtained with torch.autograd through this restated forward.
"""
import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import torch
import torch.nn.functional as F

IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


@dataclass
class PainterConfig:
    img_size: Sequence[int] = (896, 448)
    patch_size: int = 16
    embed_dim: int = 1024
    depth: int = 24
    num_heads: int = 16
    mlp_ratio: float = 4.0
    drop_path_rate: float = 0.1
    window_size: int = 14
    window_block_indexes: Sequence[int] = ()   # stock factories: effectively empty (SURVEY.md §0.1)
    pretrain_img_size: int = 224
    decoder_embed_dim: int = 64
    loss_func: str = "smoothl1"
    seggpt: bool = False
    merge_idx: int = 2
    taps: Sequence[int] = (5, 11, 17, 23)
    ln_eps: float = 1e-6

    @property
    def grid(self):
        return self.img_size[0] // self.patch_size, self.img_size[1] // self.patch_size

    def drop_path_probs(self):
        # torch.linspace(0, rate, depth) as in models_painter.py:301
        return [x.item() for x in torch.linspace(0, self.drop_path_rate, self.depth)]


def patchify(imgs, p):
    n, c, H, W = imgs.shape
    assert H == 2 * W and H % p == 0
    w = W // p
    h = 2 * w
    x = imgs.reshape(n, c, h, p, w, p).permute(0, 2, 4, 3, 5, 1)
    return x.reshape(n, h * w, p * p * c)


def unpatchify(x, p):
    n, L, D = x.shape
    w = int((L * 0.5) ** 0.5)
    h = 2 * w
    assert h * w == L
    c = D // (p * p)
    x = x.reshape(n, h, w, p, p, c).permute(0, 5, 1, 3, 2, 4)
    return x.reshape(n, c, h * p, w * p)


def patch_embed(img, weight, bias):
    """E[b,i,j,o] = bias[o] + sum_{c,r,s} W[o,c,r,s] img[b,c,16i+r,16j+s]  -> NHWC."""
    p = weight.shape[-1]
    B, C, H, W = img.shape
    h, w = H // p, W // p
    cols = img.reshape(B, C, h, p, w, p).permute(0, 2, 4, 1, 3, 5).reshape(B, h, w, C * p * p)
    return cols @ weight.reshape(weight.shape[0], -1).t() + bias


def abs_pos(pos_embed, h, w, has_cls=True):
    pe = pos_embed[:, 1:] if has_cls else pos_embed
    n = pe.shape[1]
    s = int(math.sqrt(n))
    assert s * s == n
    if s == h and s == w:
        return pe.reshape(1, h, w, -1)
    g = F.interpolate(pe.reshape(1, s, s, -1).permute(0, 3, 1, 2), size=(h, w), mode="bicubic",
                      align_corners=False)
    return g.permute(0, 2, 3, 1)


def rel_pos_lookup(rel_pos, size):
    """R[a, c] = table[a - c + size - 1]; the table is linearly resized to 2*size-1 rows if needed."""
    L = 2 * size - 1
    if rel_pos.shape[0] != L:
        t = F.interpolate(rel_pos.t().unsqueeze(0), size=L, mode="linear")[0].t()
    else:
        t = rel_pos
    ar = torch.arange(size, device=rel_pos.device)
    idx = ar[:, None] - ar[None, :] + (size - 1)
    return t[idx]  # [size, size, d]


def attention(u, sd, pre, num_heads, use_rel_pos=True):
    """u: [B, H, W, C] (already LayerNorm'ed) -> [B, H, W, C]."""
    B, H, W, C = u.shape
    N = H * W
    d = C // num_heads
    qkv = u.reshape(B, N, C) @ sd[pre + "qkv.weight"].t() + sd[pre + "qkv.bias"]
    qkv = qkv.reshape(B, N, 3, num_heads, d).permute(2, 0, 3, 1, 4)  # [3, B, nh, N, d]
    q, k, v = qkv[0], qkv[1], qkv[2]
    s = (q * d ** -0.5) @ k.transpose(-1, -2)  # [B, nh, N, N]
    if use_rel_pos:
        Rh = rel_pos_lookup(sd[pre + "rel_pos_h"], H)  # [H, H, d]
        Rw = rel_pos_lookup(sd[pre + "rel_pos_w"], W)
        rq = q.reshape(B, num_heads, H, W, d)
        rel_h = torch.einsum("bnhwc,hkc->bnhwk", rq, Rh)
        rel_w = torch.einsum("bnhwc,wkc->bnhwk", rq, Rw)
        s = (s.reshape(B, num_heads, H, W, H, W) + rel_h[..., :, None] + rel_w[..., None, :]).reshape(
            B, num_heads, N, N)
    p = s.softmax(-1)
    o = (p @ v).permute(0, 2, 1, 3).reshape(B, H, W, C)
    return o @ sd[pre + "proj.weight"].t() + sd[pre + "proj.bias"]


def _window_partition(x, ws):
    B, H, W, C = x.shape
    ph, pw = (ws - H % ws) % ws, (ws - W % ws) % ws
    x = F.pad(x, (0, 0, 0, pw, 0, ph))
    Hp, Wp = H + ph, W + pw
    x = x.reshape(B, Hp // ws, ws, Wp // ws, ws, C).permute(0, 1, 3, 2, 4, 5)
    return x.reshape(-1, ws, ws, C), (Hp, Wp)


def _window_unpartition(xw, ws, pad_hw, hw):
    Hp, Wp = pad_hw
    H, W = hw
    B = xw.shape[0] // ((Hp // ws) * (Wp // ws))
    x = xw.reshape(B, Hp // ws, Wp // ws, ws, ws, -1).permute(0, 1, 3, 2, 4, 5).reshape(B, Hp, Wp, -1)
    return x[:, :H, :W]


def feature_ensemble(a, merge):
    """SegGPT prompt ensemble on the attention output, bottom half rows only (models_seggpt.py:220-231)."""
    if merge <= 0:
        return a
    half = a.shape[1] // 2
    prompt, inputs = a[:, :half], a[:, half:]
    if merge == 1:
        P = a.shape[0] // 2
        g = inputs.reshape(2, P, *inputs.shape[1:])
        inputs = g.mean(1, keepdim=True).expand_as(g).reshape(inputs.shape)
    else:
        inputs = inputs.mean(0, keepdim=True).expand_as(inputs)
    return torch.cat([prompt, inputs], 1)


def block(z, sd, i, cfg: PainterConfig, drop=None, merge=0):
    """drop: None (eval) or (scale_attn[B'], scale_mlp[B']) with entries in {0, 1/keep}."""
    pre = f"blocks.{i}."
    C = z.shape[-1]
    u = F.layer_norm(z, (C,), sd[pre + "norm1.weight"], sd[pre + "norm1.bias"], cfg.ln_eps)
    ws = cfg.window_size if i in tuple(cfg.window_block_indexes) else 0
    if ws > 0:
        H, W = u.shape[1], u.shape[2]
        u, pad_hw = _window_partition(u, ws)
    a = attention(u, sd, pre + "attn.", cfg.num_heads)
    if ws > 0:
        a = _window_unpartition(a, ws, pad_hw, (H, W))
    a = feature_ensemble(a, merge)
    if drop is not None:
        a = a * drop[0].reshape(-1, 1, 1, 1)
    z = z + a
    v = F.layer_norm(z, (C,), sd[pre + "norm2.weight"], sd[pre + "norm2.bias"], cfg.ln_eps)
    f = F.gelu(v @ sd[pre + "mlp.fc1.weight"].t() + sd[pre + "mlp.fc1.bias"])
    f = f @ sd[pre + "mlp.fc2.weight"].t() + sd[pre + "mlp.fc2.bias"]
    if drop is not None:
        f = f * drop[1].reshape(-1, 1, 1, 1)
    return z + f


def encoder(imgs, tgts, mask, sd, cfg: PainterConfig, drops=None, seg_type=None, merge_between_batch=-1):
    x = patch_embed(imgs, sd["patch_embed.proj.weight"], sd["patch_embed.proj.bias"])
    y = patch_embed(tgts, sd["patch_embed.proj.weight"], sd["patch_embed.proj.bias"])
    B, h, w, C = x.shape
    m = mask.to(x.dtype).reshape(-1, h, w, 1)  # may broadcast over the batch (SegGPT engine passes [1, N])
    y = y * (1 - m) + sd["mask_token"] * m
    x = x + sd["segment_token_x"]
    y = y + sd["segment_token_y"]
    P = abs_pos(sd["pos_embed"], h, w)
    x = x + P
    y = y + P
    if cfg.seggpt:
        te = torch.zeros(B, 1, 1, C, dtype=x.dtype, device=x.device)
        st = seg_type.reshape(B)
        te[st == 0] = sd["type_token_cls"].reshape(1, 1, C).to(te.dtype)
        te[st == 1] = sd["type_token_ins"].reshape(1, 1, C).to(te.dtype)
        x = x + te
        y = y + te
    z = torch.cat([x, y], 0)
    taps = []
    for i in range(cfg.depth):
        merge = 0
        if cfg.seggpt and merge_between_batch >= 0 and i >= merge_between_batch:
            merge = 1 if cfg.merge_idx >= i else 2
        z = block(z, sd, i, cfg, None if drops is None else drops[i], merge)
        if i == cfg.merge_idx:
            z = (z[: z.shape[0] // 2] + z[z.shape[0] // 2:]) * 0.5
        if i in tuple(cfg.taps):
            taps.append(F.layer_norm(z, (C,), sd["norm.weight"], sd["norm.bias"], cfg.ln_eps))
    return taps


def decoder(taps, sd, cfg: PainterConfig):
    x = torch.cat(taps, -1)
    x = x @ sd["decoder_embed.weight"].t() + sd["decoder_embed.bias"]
    B, h, w, _ = x.shape
    p, c = cfg.patch_size, cfg.decoder_embed_dim
    x = x.reshape(B, h, w, p, p, c).permute(0, 5, 1, 3, 2, 4).reshape(B, c, h * p, w * p)
    x = F.conv2d(x, sd["decoder_pred.0.weight"], sd["decoder_pred.0.bias"], padding=1)
    mu = x.mean(1, keepdim=True)
    var = (x - mu).pow(2).mean(1, keepdim=True)
    x = (x - mu) / torch.sqrt(var + 1e-6)
    x = sd["decoder_pred.1.weight"][:, None, None] * x + sd["decoder_pred.1.bias"][:, None, None]
    x = F.gelu(x)
    return F.conv2d(x, sd["decoder_pred.3.weight"], sd["decoder_pred.3.bias"])


def loss_fn(pred, tgts, mask, valid, cfg: PainterConfig):
    """mask: [B or 1, N] bool.  Returns (loss, effective valid)."""
    p = cfg.patch_size
    m = mask.to(pred.dtype)[:, :, None].repeat(1, 1, p * p * 3)
    M = unpatchify(m, p)
    valid = valid.to(pred.dtype)
    if not cfg.seggpt:
        mean = torch.tensor(IMAGENET_MEAN, dtype=tgts.dtype, device=pred.device)[None, :, None, None]
        std = torch.tensor(IMAGENET_STD, dtype=tgts.dtype, device=pred.device)[None, :, None, None]
        ign = ((tgts * std + mean) * (1 - M)).sum((1, 2, 3)) < 300
        valid = valid * (~ign).to(pred.dtype)[:, None, None, None]
    Wt = M * valid
    d = pred - tgts
    if cfg.loss_func == "smoothl1":
        beta = 0.01
        l = torch.where(d.abs() < beta, 0.5 * d * d / beta, d.abs() - 0.5 * beta)
    elif cfg.loss_func == "l1":
        l = d.abs()
    elif cfg.loss_func == "l2":
        l = d * d
    elif cfg.loss_func == "l1l2":
        l = (d.abs() + d * d) * 0.5
    else:
        raise ValueError(cfg.loss_func)
    den = Wt.sum() if cfg.seggpt else Wt.sum() + 1e-2
    return (l * Wt).sum() / den


def forward(sd, cfg: PainterConfig, imgs, tgts, bool_masked_pos, valid, drops=None, seg_type=None,
            merge_between_batch=-1):
    """Returns (loss, patchify(pred) [B, N, p*p*3], mask [B(or 1), N] bool) like the reference forward
    (models_painter.py:464-472 / models_seggpt.py:471-479)."""
    h, w = imgs.shape[2] // cfg.patch_size, imgs.shape[3] // cfg.patch_size
    if bool_masked_pos is None:
        mask = torch.zeros(imgs.shape[0], h * w, dtype=torch.bool, device=imgs.device)
    else:
        mask = bool_masked_pos.flatten(1).to(torch.bool)
    taps = encoder(imgs, tgts, mask, sd, cfg, drops, seg_type, merge_between_batch)
    pred = decoder(taps, sd, cfg)
    loss = loss_fn(pred, tgts, mask, valid, cfg)
    return loss, patchify(pred, cfg.patch_size), mask


def draw_drop_scales(cfg: PainterConfig, B, dtype=torch.float32, generator=None):
    """Per-block DropPath scales, drawn in the reference's order (attn branch then mlp branch, batch 2B for
    blocks <= merge_idx; block 0 has p=0 -> nn.Identity, no draw).  Entries are in {0, 1/keep}."""
    out = []
    for i, p in enumerate(cfg.drop_path_probs()):
        Bp = 2 * B if i <= cfg.merge_idx else B
        if p == 0.0:
            out.append((torch.ones(Bp, dtype=dtype), torch.ones(Bp, dtype=dtype)))
            continue
        keep = 1 - p
        pair = []
        for _ in range(2):
            r = (keep + torch.rand((Bp, 1, 1, 1), dtype=dtype, generator=generator)).floor_()
            pair.append((r / keep).reshape(Bp))
        out.append(tuple(pair))
    return out
