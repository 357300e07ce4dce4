"""Kernel contracts at the model's shapes, element by element.

- Every GEMM epilogue on both tensor-core kernels (single CTA with 128-row tiles, gemm.cu; CTA pairs with 256-row
  tiles, gemm2.cu), at the N and K of every call site of engine.py and accurate.py and the token counts the model
  produces, with the default plan and with every legal forced tile.
- The epilogue GELU / GELU' over every finite bf16 input with |z| <= 12.
- The shape limits of the attention and decoder-head kernels: every accepted limit computes correctly, and the
  shapes just past it are refused on the host before any launch.

The reference is plain torch on the same bf16 operands in fp64.  The bound of one element scales with what went into
it, S = |alpha| |A| |B|^T + |bias| (+ |aux|): fp32 outputs 1e-5 S; bf16 outputs one bf16 ulp of the reference value
plus 1e-5 S.  Every output buffer is pre-filled with NaN and is larger than the output (extra rows past M, extra
columns around a column slice): afterwards every element the call owns must hold its value and every other element
must still be NaN.
"""
import contextlib
import ctypes
import math
from collections import namedtuple

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"
NAN = float("nan")

EPI_BF16, EPI_F32, EPI_GELU, EPI_RESID, EPI_DGELU, EPI_PIXSHUF = range(6)
KIND_NAMES = {EPI_BF16: "bf16", EPI_F32: "f32", EPI_GELU: "gelu", EPI_RESID: "resid", EPI_DGELU: "dgelu",
              EPI_PIXSHUF: "pixshuf"}

# ------------------------------------------------------------------------------------------------------------------
# GEMM case table (also read by test_kernel_contract_coverage.py, without a GPU)
# ------------------------------------------------------------------------------------------------------------------
# Token counts (the GEMMs' M, the weight gradients' K): B=1 at 896x448 after / before the early merge, B=8, B=1 at
# 1792x896, one count whose last 256-row tile is more than half full (400 = 256 + 144) and one below 256.
TOKENS = (1568, 3136, 12544, 6272, 400, 200)
FEW = (3136, 400, 200)
ROWS_PER_SAMPLE = 1568                         # DropPath row groups: one sample's tokens at 896x448
ROWSCALE_PATTERN = (1.0, 0.0, 1.25, 0.5, 0.0, 1.0, 0.75, 2.0)
# EPI_PIXSHUF token grid (h, w) per token count: p = 16, c = 64, so M = B * h * w
PIXSHUF_GRID = {1568: (56, 28), 3136: (56, 28), 12544: (56, 28), 6272: (112, 56), 400: (20, 20), 200: (10, 20)}


def _pad64(n):
    return (n + 63) // 64 * 64


Site = namedtuple("Site", "name kind mnk ta tb bias alpha acc rowscale tokens")


def _site(name, kind, mnk, ta=False, tb=False, bias=False, alpha=1.0, acc=0, rowscale=False, tokens=TOKENS):
    return Site(name, kind, mnk, ta, tb, bias, alpha, acc, rowscale, tokens)


SITES = [
    # forward (engine.py EmbedFn / BlockFn.forward / DecoderFn.forward)
    _site("patch_embed", EPI_F32, lambda T: (T, 1024, 768), bias=True),
    _site("qkv", EPI_BF16, lambda T: (T, 3072, 1024), bias=True),
    _site("qkv_alpha", EPI_BF16, lambda T: (T, 3072, 1024), bias=True, alpha=0.5, tokens=FEW),
    _site("proj_resid", EPI_RESID, lambda T: (T, 1024, 1024), bias=True, rowscale=True),
    _site("proj_window", EPI_F32, lambda T: (T, 1024, 1024), bias=True, tokens=FEW),
    _site("proj_alpha", EPI_F32, lambda T: (T, 1024, 1024), bias=True, alpha=0.5, tokens=FEW),
    _site("fc1", EPI_GELU, lambda T: (T, 4096, 1024), bias=True),
    _site("fc1_nobias", EPI_GELU, lambda T: (T, 4096, 1024), tokens=FEW),
    _site("fc2_resid", EPI_RESID, lambda T: (T, 1024, 4096), bias=True, rowscale=True),
    _site("fc2_resid_alpha", EPI_RESID, lambda T: (T, 1024, 4096), bias=True, rowscale=True, alpha=0.5, tokens=FEW),
    _site("decoder_embed", EPI_PIXSHUF, lambda T: (T, 16384, 4096), bias=True),
    _site("decoder_embed_nobias", EPI_PIXSHUF, lambda T: (T, 16384, 4096), tokens=(3136, 200)),
    # backward: dgrad (B read MN-major) and wgrad (both operands MN-major, zero-initialised fp32 output)
    _site("fc2_dgrad", EPI_DGELU, lambda T: (T, 4096, 1024), tb=True),
    _site("fc2_dgrad_bias", EPI_DGELU, lambda T: (T, 4096, 1024), tb=True, bias=True, tokens=FEW),
    _site("fc1_dgrad", EPI_BF16, lambda T: (T, 1024, 4096), tb=True),
    _site("proj_dgrad", EPI_BF16, lambda T: (T, 1024, 1024), tb=True, tokens=FEW),
    _site("qkv_dgrad", EPI_BF16, lambda T: (T, 1024, 3072), tb=True),
    _site("qkv_dgrad_window", EPI_F32, lambda T: (T, 1024, 3072), tb=True),
    _site("qkv_dgrad_accumulate", EPI_F32, lambda T: (T, 1024, 3072), tb=True, acc=1, tokens=FEW),
    _site("dcat_dgrad", EPI_BF16, lambda T: (T, 4096, 16384), tb=True, tokens=(1568, 3136, 400, 200)),
    _site("fc1_wgrad", EPI_F32, lambda T: (4096, 1024, T), ta=True, tb=True, acc=2),
    _site("qkv_wgrad", EPI_F32, lambda T: (3072, 1024, T), ta=True, tb=True, acc=2),
    _site("proj_wgrad", EPI_F32, lambda T: (1024, 1024, T), ta=True, tb=True, acc=2, tokens=FEW),
    _site("decoder_embed_wgrad", EPI_F32, lambda T: (16384, 4096, T), ta=True, tb=True, acc=2, tokens=(1568, 400)),
    _site("fc1_accumulate", EPI_F32, lambda T: (4096, 1024, T), ta=True, tb=True, acc=1, alpha=0.5, tokens=FEW),
    # fp32-accurate mode (accurate.py): K = 6 x the fp32 K, P.V into a 64-column slice of the attention output
    _site("accurate_qkv", EPI_F32, lambda T: (T, 3072, 6144), bias=True, tokens=FEW),
    _site("accurate_pv", EPI_F32, lambda T: (T, 64, 6 * _pad64(T)), tb=True, tokens=(1568, 6272, 400, 200)),
    _site("accurate_resid", EPI_RESID, lambda T: (T, 1024, 6144), bias=True, tokens=FEW),
    _site("resid_nobias", EPI_RESID, lambda T: (T, 1024, 1024), rowscale=True, tokens=FEW),
]

# (pk_gemm_use_2cta, pk_gemm_force_bn): the default plan, the single-CTA kernel at every tile width, the CTA-pair
# kernel at both of its tile widths.  The default is the library's own setting (CTA pairs on, heuristic BN).
HOOKS = ((1, 0), (0, 64), (0, 128), (0, 256), (1, 128), (1, 256))


def gemm_cases():
    """(site, token count) pairs of the GEMM test."""
    return [(s, T) for s in SITES for T in s.tokens]


def hooks_for(N):
    """The hook settings that are legal for an output width N (a forced BN must divide N)."""
    return [(pair, bn) for pair, bn in HOOKS if bn == 0 or N % bn == 0]


def plan(M, N, K, kind, acc):
    """pk_gemm_plan under the current hooks: dict(pair, BN, ...)."""
    from painter_b200 import _lib
    L = _lib.lib()
    out = (ctypes.c_int * 9)()
    assert L.pk_gemm_plan(M, N, K, kind, acc, out) == 0, L.pk_last_error()
    keys = ["pair", "BN", "mt", "nt", "splits", "kbps", "sk_units", "group_m", "workers"]
    return dict(zip(keys, list(out)))


@contextlib.contextmanager
def gemm_hooks(pair, bn):
    from painter_b200 import _lib
    L = _lib.lib()
    L.pk_gemm_use_2cta(pair)
    L.pk_gemm_force_bn(bn)
    try:
        yield
    finally:
        L.pk_gemm_force_bn(0)
        L.pk_gemm_use_2cta(1)


def expected_kernel(M, N, pair, bn):
    """(pair, BN) a forced hook setting must produce, or None for the default plan."""
    if bn == 0:
        return None
    return (1 if (pair and bn in (128, 256) and M >= 256) else 0), bn


# ------------------------------------------------------------------------------------------------------------------
# element-wise checks
# ------------------------------------------------------------------------------------------------------------------
def bf16_ulp(x):
    """One bf16 ulp of |x| (8 significant bits), fp64."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), e - 8)


def gelu64(z):
    return z * 0.5 * torch.erfc(-z / math.sqrt(2.0))


def gelu_grad64(z):
    return 0.5 * torch.erfc(-z / math.sqrt(2.0)) + z * torch.exp(-0.5 * z * z) / math.sqrt(2.0 * math.pi)


def assert_close(got, ref, bound, what):
    """|got - ref| <= bound element by element (a NaN in got fails)."""
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        idx = bad.nonzero()[0].tolist()
        ratio = (err / bound).nan_to_num(nan=float("inf")).max().item()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bounds; first at {idx}: got "
                             f"{got[tuple(idx)].item()!r} want {ref[tuple(idx)].item()!r} bound "
                             f"{bound[tuple(idx)].item():.3g}; worst err/bound {ratio:.3g}")


class Sentinel:
    """NaN-filled buffer with a [rows, cols] view at (0, col0): `pad_rows` rows past the view and `pad_cols` columns
    around it (first col0 of them to its left) belong to nobody."""

    def __init__(self, rows, cols, dtype, pad_rows=256, pad_cols=0, col0=0):
        self.buf = torch.full((rows + pad_rows, cols + pad_cols), NAN, dtype=dtype, device=DEV)
        self.rows, self.cols, self.col0 = rows, cols, col0
        self.view = self.buf[:rows, col0:col0 + cols]

    def assert_untouched_outside(self, what):
        b, r, c0, c1 = self.buf, self.rows, self.col0, self.col0 + self.cols
        for name, part in (("rows past the output", b[r:]), ("columns left of the output", b[:r, :c0]),
                           ("columns right of the output", b[:r, c1:])):
            if part.numel():
                assert bool(torch.isnan(part).all()), f"{what}: a store landed in the {name}"


def _operand(rows, cols, strided, scale, gen):
    """bf16 [rows, cols] operand; strided: a column slice of a wider matrix (leading dimension cols + 64)."""
    x = (torch.randn(rows, cols + (64 if strided else 0), generator=gen, device=DEV) * scale).bfloat16()
    return x[:, :cols] if strided else x


def _rowscale_rows(M, rowscale):
    return rowscale.double().repeat_interleave(ROWS_PER_SAMPLE)[:M]


@pytest.fixture(autouse=True)
def _fp32_references():
    """References in plain fp32 must not use TF32 (torch's default for convolutions)."""
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


# ------------------------------------------------------------------------------------------------------------------
# 1. GEMM: every epilogue on both kernels
# ------------------------------------------------------------------------------------------------------------------
def _run_site(site, M, N, K, ops_in, strided):
    """One pk_gemm_bf16 call of `site` into fresh NaN sentinels; returns (sentinels, output views)."""
    from painter_b200 import ops
    a, b, bias, aux, rowscale, init = ops_in
    kind = site.kind
    pad = dict(pad_cols=96, col0=32) if strided else {}
    if kind == EPI_PIXSHUF:
        h, w = PIXSHUF_GRID[M]
        Bs = M // (h * w)
        n = Bs * h * 16 * w * 16 * 64
        s = Sentinel(1, n, torch.bfloat16, pad_rows=0, pad_cols=4096)
        out = s.view.view(Bs, h * 16, w * 16, 64)
        ops.gemm(a, b, trans_a=site.ta, trans_b=site.tb, kind=kind, bias=bias, alpha=site.alpha,
                 pixshuf=(h, w, 16, 64, out))
        return [s], [out]
    odt = torch.float32 if kind in (EPI_F32, EPI_RESID) else torch.bfloat16
    s = Sentinel(M, N, odt, **pad)
    if init is not None:
        s.view.copy_(init)
    sents, outs = [s], [s.view]
    out2 = None
    if kind == EPI_GELU:
        s2 = Sentinel(M, N, torch.bfloat16, **pad)
        sents.append(s2)
        outs.append(s2.view)
        out2 = s2.view
    if aux is not None and strided:      # ld_aux != ldc
        wide = torch.full((M, N + 160), NAN, dtype=aux.dtype, device=DEV)
        wide[:, 8:8 + N] = aux
        aux = wide[:, 8:8 + N]
    ops.gemm(a, b, trans_a=site.ta, trans_b=site.tb, kind=kind, out=s.view, out2=out2, bias=bias, aux=aux,
             rowscale=rowscale, rows_per_group=ROWS_PER_SAMPLE if rowscale is not None else 0, alpha=site.alpha,
             accumulate=site.acc)
    return sents, outs


def _check_site(site, M, N, outs, ref, what):
    """ref: dict of fp64 tensors from _site_reference."""
    kind = site.kind
    if kind == EPI_PIXSHUF:
        h, w = PIXSHUF_GRID[M]
        Bs = M // (h * w)

        def shuffle(t):   # models_painter.py: 'nhwpqc->nchpwq', then NHWC
            t = torch.einsum("nhwpqc->nchpwq", t.reshape(Bs, h, w, 16, 16, 64))
            return t.reshape(Bs, 64, h * 16, w * 16).permute(0, 2, 3, 1)

        pre, S = shuffle(ref["pre"]), shuffle(ref["S"])
        assert_close(outs[0], pre, bf16_ulp(pre) + 1e-5 * S, what)
        return
    out = outs[0]
    pre, S = ref["pre"], ref["S"]
    if kind == EPI_BF16:
        assert_close(out, pre, bf16_ulp(pre) + 1e-5 * S, what)
    elif kind == EPI_F32:
        assert_close(out, ref["want"], 1e-5 * ref["S_out"], what)
    elif kind == EPI_RESID:
        assert_close(out, ref["want"], 1e-5 * ref["S_out"], what)
        zero = ref["zero_rows"]
        if zero is not None and bool(zero.any()):
            assert torch.equal(out[zero], ref["aux"][zero]), f"{what}: rows scaled by 0 differ from aux"
    elif kind == EPI_GELU:
        assert_close(out, pre, bf16_ulp(pre) + 1e-5 * S, what + " (z)")
        g = gelu64(out.double())
        assert_close(outs[1], g, bf16_ulp(g) + 2.0 ** -15, what + " (gelu(z))")
    elif kind == EPI_DGELU:
        want = ref["want"]
        assert_close(out, want, bf16_ulp(want) + 2.0 ** -13 * pre.abs() + 1.2e-5 * S, what)


def _site_inputs(site, M, N, K, strided, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    a = _operand(K, M, strided, 1.0, gen) if site.ta else _operand(M, K, strided, 1.0, gen)
    # weight-like B; for the GELU epilogues z = acc + bias spreads over about [-8, 8]
    bs = 2.0 / math.sqrt(K)
    b = _operand(K, N, strided, bs, gen) if site.tb else _operand(N, K, strided, bs, gen)
    bias = torch.randn(N, generator=gen, device=DEV) if site.bias else None
    aux = None
    if site.kind == EPI_RESID:
        aux = torch.randn(M, N, generator=gen, device=DEV)
    elif site.kind == EPI_DGELU:
        aux = (torch.randn(M, N, generator=gen, device=DEV) * 2).bfloat16()
    rowscale = None
    if site.rowscale:
        G = (M + ROWS_PER_SAMPLE - 1) // ROWS_PER_SAMPLE
        rowscale = torch.tensor([ROWSCALE_PATTERN[i % len(ROWSCALE_PATTERN)] for i in range(G)], device=DEV)
    init = None
    if site.acc == 1:
        init = torch.randn(M, N, generator=gen, device=DEV)
    elif site.acc == 2:
        init = torch.zeros(M, N, device=DEV)
    return a, b, bias, aux, rowscale, init


def _site_reference(site, M, inputs):
    a, b, bias, aux, rowscale, init = inputs
    A = (a.t() if site.ta else a).double()
    B = (b.t() if site.tb else b).double()
    acc = A @ B.t()
    S = abs(site.alpha) * (A.abs() @ B.abs().t())
    del A, B
    pre = site.alpha * acc
    if bias is not None:
        pre += bias.double()
        S += bias.double().abs()
    ref = {"pre": pre, "S": S}
    if site.kind == EPI_F32:
        ref["want"] = pre + init.double() if init is not None else pre
        ref["S_out"] = S + init.double().abs() if init is not None else S
    elif site.kind == EPI_RESID:
        rs = _rowscale_rows(M, rowscale)[:, None] if rowscale is not None else 1.0
        ref["want"] = aux.double() + rs * pre
        ref["S_out"] = aux.double().abs() + (rs.abs() * S if rowscale is not None else S)
        ref["aux"] = aux
        ref["zero_rows"] = (_rowscale_rows(M, rowscale) == 0) if rowscale is not None else None
    elif site.kind == EPI_DGELU:
        ref["want"] = pre * gelu_grad64(aux.double())
        ref["S"] = S * 1.2      # |gelu'| < 1.13
    return ref


@pytest.mark.parametrize("site,T", gemm_cases(), ids=[f"{s.name}-T{T}" for s, T in gemm_cases()])
def test_gemm_epilogue_on_both_kernels(site, T):
    M, N, K = site.mnk(T)
    cache = {}
    for i, (pair, bn) in enumerate(hooks_for(N)):
        strided = i % 2 == 1     # every other setting: A, B, out, out2 and aux as slices of wider buffers
        if strided not in cache:
            inputs = _site_inputs(site, M, N, K, strided, seed=T + 7 * int(strided))
            cache[strided] = inputs, _site_reference(site, M, inputs)
        inputs, ref = cache[strided]
        with gemm_hooks(pair, bn):
            p = plan(M, N, K, site.kind, site.acc)
            want = expected_kernel(M, N, pair, bn)
            what = (f"{site.name} M={M} N={N} K={K} {'cta-pair' if p['pair'] else 'single-cta'} BN={p['BN']} "
                    f"(hooks 2cta={pair} bn={bn}, {'strided' if strided else 'dense'})")
            if want is not None:
                assert (p["pair"], p["BN"]) == want, what
            sents, outs = _run_site(site, M, N, K, inputs, strided)
        torch.cuda.synchronize()
        for s in sents:
            s.assert_untouched_outside(what)
        _check_site(site, M, N, outs, ref, what)
        del sents, outs


def test_gemm_stream_k_under_sm_budget_matches_unbudgeted():
    """pk_set_sm_budget (the multi-GPU backward leaves SMs to NCCL) re-partitions the stream-K units of a weight
    gradient over fewer clusters; the result must not change beyond fp32 summation order."""
    from painter_b200 import ops
    site = next(s for s in SITES if s.name == "fc1_wgrad")
    M, N, K = site.mnk(12544)
    inputs = _site_inputs(site, M, N, K, False, seed=11)
    ref = _site_reference(site, M, inputs)
    free = plan(M, N, K, EPI_F32, 2)
    old = ops.set_sm_budget(132)
    try:
        capped = plan(M, N, K, EPI_F32, 2)
        s_cap, o_cap = _run_site(site, M, N, K, inputs, False)
    finally:
        ops.set_sm_budget(old)
    assert plan(M, N, K, EPI_F32, 2) == free
    assert capped["pair"] == 1 and capped["sk_units"] > 0 and capped["workers"] <= 66
    assert capped["sk_units"] != free["sk_units"] or capped["workers"] != free["workers"]
    s_free, o_free = _run_site(site, M, N, K, inputs, False)
    torch.cuda.synchronize()
    for s in s_cap + s_free:
        s.assert_untouched_outside("stream-K")
    _check_site(site, M, N, o_cap, ref, "stream-K under a 132-SM budget")
    _check_site(site, M, N, o_free, ref, "stream-K on all SMs")
    assert_close(o_cap[0], o_free[0].double(), 2e-5 * ref["S_out"], "budgeted vs unbudgeted")


# ------------------------------------------------------------------------------------------------------------------
# 2. GELU / GELU' of the epilogue over every bf16 input
# ------------------------------------------------------------------------------------------------------------------
GELU_RANGES = ((-12.0, -6.0), (-6.0, -4.0), (-4.0, -3.0), (-3.0, -2.0), (-2.0, 0.0), (0.0, 12.01))


def all_bf16_upto(limit):
    """Every finite bf16 value z with |z| <= limit (both zeros included), fp32."""
    bits = torch.arange(0, 1 << 16, dtype=torch.int32).to(torch.int16)
    z = bits.view(torch.bfloat16).float()
    return z[torch.isfinite(z) & (z.abs() <= limit)]


def _identity_gemm_operands(values, fill):
    """A = I (512 x 512) and B [128, 512] with B^T holding `values` (rest `fill`): then acc = B^T exactly."""
    M = K = 512
    N = 128
    assert values.numel() <= M * N
    flat = torch.full((M * N,), fill, dtype=torch.float32)
    flat[:values.numel()] = values
    bt = flat.view(M, N).bfloat16().to(DEV)           # acc[m, n] = B[n, m]
    a = torch.eye(M, K, device=DEV).bfloat16()
    return a, bt.t().contiguous(), bt, values.numel()


GELU_HOOKS = ((0, 64), (0, 128), (1, 128))


def gelu_errors(z, got, want, extra):
    """Worst |got - want| / (ulp(want) + extra) and worst error in ulps of want, per range of z."""
    err = (got.double() - want).abs()
    rows = []
    for lo, hi in GELU_RANGES:
        m = (z >= lo) & (z < hi)
        ratio = (err[m] / (bf16_ulp(want[m]) + extra[m])).max().item()
        ulps = (err[m] / bf16_ulp(want[m])).max().item()
        rows.append((lo, hi, ratio, ulps))
    return rows


def _fmt(rows):
    return "; ".join(f"[{lo:g},{hi:g}): bound ratio {r:.3g}, {u:.3g} ulp" for lo, hi, r, u in rows)


def test_gelu_epilogue_over_every_bf16_input():
    """EPI_GELU with acc = every bf16 z: |gelu(z) - gelu_erf(z)| <= 1 bf16 ulp of the true value + 2^-15."""
    from painter_b200 import ops
    zs = all_bf16_upto(12.0)
    a, b, bt, n = _identity_gemm_operands(zs, 0.0)
    for pair, bn in GELU_HOOKS:
        with gemm_hooks(pair, bn):
            p = plan(512, 128, 512, EPI_GELU, 0)
            assert (p["pair"], p["BN"]) == expected_kernel(512, 128, pair, bn)
            z, h = ops.gemm(a, b, kind=EPI_GELU)
        assert torch.equal(z, bt), "the identity GEMM must reproduce B^T exactly"
        zf = z.double().flatten()[:n]
        want = gelu64(zf)
        got = h.flatten()[:n]
        rows = gelu_errors(zf, got, want, torch.full_like(want, 2.0 ** -15))
        assert max(r[2] for r in rows) <= 1.0, f"{'cta-pair' if p['pair'] else 'single-cta'} BN={bn}: {_fmt(rows)}"


@pytest.mark.parametrize("c", [1.0, -3.0, 0.375, 96.0])
def test_dgelu_epilogue_over_every_bf16_input(c):
    """EPI_DGELU with aux = every bf16 z and acc = c: |out - c gelu'(z)| <= 1 bf16 ulp + |c| 2^-13."""
    from painter_b200 import ops
    zs = all_bf16_upto(12.0)
    _, _, zt, n = _identity_gemm_operands(zs, 0.0)          # aux [512, 128] = z
    a = torch.eye(512, device=DEV).bfloat16()
    b = torch.full((128, 512), c, device=DEV).bfloat16()    # acc = c everywhere
    for pair, bn in GELU_HOOKS:
        with gemm_hooks(pair, bn):
            p = plan(512, 128, 512, EPI_DGELU, 0)
            assert (p["pair"], p["BN"]) == expected_kernel(512, 128, pair, bn)
            out = ops.gemm(a, b, kind=EPI_DGELU, aux=zt)
        zf = zt.double().flatten()[:n]
        want = c * gelu_grad64(zf)
        rows = gelu_errors(zf, out.flatten()[:n], want, torch.full_like(want, abs(c) * 2.0 ** -13))
        assert max(r[2] for r in rows) <= 1.0, f"{'cta-pair' if p['pair'] else 'single-cta'} BN={bn}: {_fmt(rows)}"


# ------------------------------------------------------------------------------------------------------------------
# 3. Attention: the accepted limits compute correctly, the shapes past them are refused before any launch
# ------------------------------------------------------------------------------------------------------------------
def relmax(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-12)).item()


def _table(L, Lpad, gen):
    """bf16 rel-pos table [Lpad, 64]: L random rows, zero rows after them."""
    t = torch.zeros(Lpad, 64, device=DEV)
    t[:L] = torch.randn(L, 64, generator=gen, device=DEV) * 0.3
    return t.bfloat16()


def _attn_reference(qkv, th, tw, B, heads, h, w):
    """(out [B*N, C], lse [B*heads, N] in the log2 domain): models_painter.py:73-86 + vitdet_utils.py:96-125."""
    N, C = h * w, heads * 64
    q, k, v = qkv.reshape(B, N, 3, heads, 64).permute(2, 0, 3, 1, 4)
    s = (q * 0.125) @ k.transpose(-1, -2)
    ih = torch.arange(h, device=DEV)[:, None] - torch.arange(h, device=DEV)[None, :] + h - 1
    iw = torch.arange(w, device=DEV)[:, None] - torch.arange(w, device=DEV)[None, :] + w - 1
    rq = q.reshape(B, heads, h, w, 64)
    rel_h = torch.einsum("bnhwc,hkc->bnhwk", rq, th[ih])
    rel_w = torch.einsum("bnhwc,wkc->bnhwk", rq, tw[iw])
    s = (s.reshape(B, heads, h, w, h, w) + rel_h[..., :, None] + rel_w[..., None, :]).reshape(B, heads, N, N)
    lse = torch.logsumexp(s, -1) / math.log(2.0)
    return (s.softmax(-1) @ v).permute(0, 2, 1, 3).reshape(B * N, C), lse.reshape(B * heads, N)


# (B, heads, h, w, extra zero table rows, backward too)
ATTN_SHAPES = [
    (2, 2, 16, 8, 0, True),      # w = 8
    (1, 1, 112, 8, 0, True),     # the backward's height limit: th_pad = 224
    (1, 1, 128, 8, 0, False),    # the forward's height limit: th_pad = 256
    (1, 1, 128, 56, 0, False),   # both forward limits: th_pad = 256, tw_pad = 112
    (2, 16, 14, 14, 0, True),    # windowed-block geometry
    (2, 2, 14, 14, 32, True),    # tables padded past pad16(2L - 1)
]


@pytest.mark.parametrize("B,heads,h,w,extra,bwd", ATTN_SHAPES)
def test_attention_accepted_limits(B, heads, h, w, extra, bwd):
    from painter_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(h * 100 + w)
    N, C = h * w, heads * 64
    qkv = (torch.randn(B * N, 3 * C, generator=gen, device=DEV) * 1.5).bfloat16()
    pad16 = lambda n: (n + 15) // 16 * 16
    th = _table(2 * h - 1, pad16(2 * h - 1) + extra, gen)
    tw = _table(2 * w - 1, pad16(2 * w - 1) + extra, gen)
    out, lse = ops.attn_fwd(qkv, th, tw, B, heads, h, w)
    q64 = qkv.double().requires_grad_(bwd)
    t64, w64 = th.double().requires_grad_(bwd), tw.double().requires_grad_(bwd)
    ro, rlse = _attn_reference(q64, t64, w64, B, heads, h, w)
    assert relmax(out, ro) < 1e-2
    assert (lse.double() - rlse).abs().max().item() < 1e-3, "lse"
    if w == 8:   # the training forward keeps the bias rows: same results
        out2, lse2, rel = ops.attn_fwd(qkv, th, tw, B, heads, h, w, save_rel=True)
        assert torch.equal(out2, out) and torch.equal(lse2, lse)
    if not bwd:
        return
    dout = (torch.randn(B * N, C, generator=gen, device=DEV) * 0.5).bfloat16()
    (ro * dout.double()).sum().backward()
    dqkv, dTh, dTw = ops.attn_bwd(qkv, out, dout, lse, th, tw, B, heads, h, w)
    g, d = q64.grad.reshape(B * N, 3, C), dqkv.reshape(B * N, 3, C)
    for i in range(3):
        assert relmax(d[:, i], g[:, i]) < 2e-2, "qkv"[i]
    assert relmax(dTh, t64.grad[:2 * h - 1]) < 2e-2 and relmax(dTw, w64.grad[:2 * w - 1]) < 2e-2
    # dT_out accumulates into running table gradients
    acc_h = torch.randn(2 * h - 1, 64, generator=gen, device=DEV)
    acc_w = torch.randn(2 * w - 1, 64, generator=gen, device=DEV)
    h0, w0 = acc_h.clone(), acc_w.clone()
    ops.attn_bwd(qkv, out, dout, lse, th, tw, B, heads, h, w, dT_out=(acc_h, acc_w))
    assert relmax(acc_h - h0, dTh) < 1e-4 and relmax(acc_w - w0, dTw) < 1e-4
    if w == 8:
        dqkv2, dTh2, dTw2 = ops.attn_bwd(qkv, out2, dout, lse2, th, tw, B, heads, h, w, rel=rel)
        d2 = dqkv2.reshape(B * N, 3, C)
        for i in range(3):
            assert relmax(d2[:, i], d[:, i]) < 2e-3, "saved vs recomputed " + "qkv"[i]
        assert relmax(dTh2, dTh) < 1e-3 and relmax(dTw2, dTw) < 1e-3


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, NAN, dtype=dtype, device=DEV)


def _attn_fwd_refused(B, heads, h, w, th_pad, tw_pad):
    """pk_attn_fwd on a shape its host checks refuse: (message, outputs untouched)."""
    from painter_b200 import _lib
    L = _lib.lib()
    N, C = h * w, heads * 64
    qkv = torch.zeros(B * N, 3 * C, dtype=torch.bfloat16, device=DEV)
    th = torch.zeros(th_pad, 64, dtype=torch.bfloat16, device=DEV)
    tw = torch.zeros(tw_pad, 64, dtype=torch.bfloat16, device=DEV)
    out, lse = _nan(B * N, C, dtype=torch.bfloat16), _nan(B * heads, N)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = L.pk_attn_fwd(vp(qkv), vp(th), vp(tw), vp(out), vp(lse), B, heads, h, w, th_pad, tw_pad,
                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert rc != 0, f"pk_attn_fwd accepted h={h} w={w} th_pad={th_pad} tw_pad={tw_pad}"
    return L.pk_last_error().decode(), bool(torch.isnan(out.float()).all() and torch.isnan(lse).all())


def _attn_bwd_refused(B, heads, h, w, th_pad, tw_pad):
    from painter_b200 import _lib
    L = _lib.lib()
    L.pk_attn_bwd_ws_floats.restype = ctypes.c_longlong
    N, C = h * w, heads * 64
    Np = (N + 127) // 128 * 128
    qkv = torch.zeros(B * N, 3 * C, dtype=torch.bfloat16, device=DEV)
    O = torch.zeros(B * N, C, dtype=torch.bfloat16, device=DEV)
    dO = torch.zeros(B * N, C, dtype=torch.bfloat16, device=DEV)
    lse = torch.zeros(B * heads, N, device=DEV)
    th = torch.zeros(th_pad, 64, dtype=torch.bfloat16, device=DEV)
    tw = torch.zeros(tw_pad, 64, dtype=torch.bfloat16, device=DEV)
    dqkv = _nan(B * N, 3 * C, dtype=torch.bfloat16)
    dTh, dTw, delta = _nan(max(2 * h - 1, 1), 64), _nan(max(2 * w - 1, 1), 64), _nan(B * heads * N)
    relh, relw = _nan(B * heads * Np * h), _nan(B * heads * Np * w)
    ws = _nan(max(int(L.pk_attn_bwd_ws_floats(B, heads, h, w)), 1))
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = L.pk_attn_bwd(vp(qkv), vp(O), vp(dO), vp(lse), vp(th), vp(tw), vp(dqkv), vp(dTh), vp(dTw), vp(delta),
                       vp(relh), vp(relw), vp(ws), B, heads, h, w, th_pad, tw_pad,
                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert rc != 0, f"pk_attn_bwd accepted h={h} w={w} th_pad={th_pad} tw_pad={tw_pad}"
    untouched = all(bool(torch.isnan(t.float()).all()) for t in (dqkv, dTh, dTw, delta, relh, relw))
    return L.pk_last_error().decode(), untouched


def test_attention_refuses_shapes_past_its_limits():
    msg, untouched = _attn_fwd_refused(1, 1, 4, 3, 16, 16)
    assert "width 3" in msg and untouched, msg
    msg, untouched = _attn_fwd_refused(1, 1, 8, 8, 272, 16)
    assert "th_pad=272" in msg and untouched, msg
    msg, untouched = _attn_fwd_refused(1, 1, 8, 8, 16, 128)
    assert "tw_pad=128" in msg and untouched, msg
    msg, untouched = _attn_bwd_refused(1, 1, 4, 3, 16, 16)
    assert "width 3" in msg and untouched, msg
    msg, untouched = _attn_bwd_refused(1, 1, 8, 8, 240, 16)
    assert "th_pad=240" in msg and untouched, msg
    # the forward runs up to h = 128, the backward only up to h = 112 (th_pad <= 224)
    for h in range(113, 129):
        th_pad = (2 * h - 1 + 15) // 16 * 16
        msg, untouched = _attn_bwd_refused(1, 1, h, 8, th_pad, 16)
        assert f"th_pad={th_pad}" in msg and untouched, (h, msg)


# ------------------------------------------------------------------------------------------------------------------
# 4. Decoder head: conv3x3 -> LayerNorm2D -> GELU -> conv1x1 -> loss, and the conv's two gradients
# ------------------------------------------------------------------------------------------------------------------
P = 16
IMNET_MEAN, IMNET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
# (B, H, W): the full 896x448 size (the wgrad splits over many CTAs) and W = 32 (32 x 4 conv tiles)
DECODER_GEOMETRIES = [(2, 896, 448), (2, 64, 32)]


def _loss_terms(d, kind):
    ad = d.abs()
    if kind == 0:
        return torch.where(ad < 0.01, 0.5 * d * d / 0.01, ad - 0.005)
    if kind == 1:
        return ad
    if kind == 2:
        return d * d
    return 0.5 * (ad + d * d)


def _decoder_inputs(B, H, W, seed, maskB):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda *s, sc=1.0: torch.randn(*s, generator=gen, device=DEV) * sc
    g = r(B, H, W, 64).bfloat16()
    c3w = r(64, 64, 3, 3, sc=0.05)
    c3b, lnw, lnb = r(64, sc=0.1), 1 + r(64, sc=0.1), r(64, sc=0.1)
    c1w, c1b = r(3, 64, 1, 1, sc=0.2), r(3, sc=0.1)
    tgts = r(B, 3, H, W)
    mask = (torch.rand(maskB, (H // P) * (W // P), generator=gen, device=DEV) < 0.5).to(torch.uint8)
    valid = torch.ones(B, 3, H, W, device=DEV)
    valid[torch.rand(B, 3, H, W, generator=gen, device=DEV) < 0.1] = 0
    valid[torch.rand(B, 3, H, W, generator=gen, device=DEV) > 0.95] = 10
    hp = torch.cat([c3b, lnw, lnb, c1w.reshape(-1), c1b, torch.zeros(5, device=DEV)])
    return g, c3w, hp, tgts, mask, valid


def _head_from_c1(c1_nhwc, hp):
    """fp64 LayerNorm2D + exact GELU + conv1x1 of the stored (bf16) conv output -> pred [B, 3, H, W] and the
    per-element magnitude of the pred sums."""
    x = c1_nhwc.permute(0, 3, 1, 2)
    lnw, lnb = hp[64:128].double(), hp[128:192].double()
    c1w, c1b = hp[192:384].double().view(3, 64), hp[384:387].double()
    mu = x.mean(1, keepdim=True)
    xh = (x - mu) / torch.sqrt((x - mu).pow(2).mean(1, keepdim=True) + 1e-6)
    ge = gelu64(lnw[:, None, None] * xh + lnb[:, None, None])
    pred = torch.einsum("ok,bkhw->bohw", c1w, ge) + c1b[:, None, None]
    mag = torch.einsum("ok,bkhw->bohw", c1w.abs(), ge.abs() + lnw.abs()[:, None, None] * (xh.abs() + 1)) + c1b.abs()[:, None, None]
    return pred, mag


def _mask_pixels(mask, B, H, W):
    """[maskB, N] token mask -> [B, 3, H, W] (the reference's patch mask, broadcast over samples when maskB = 1)."""
    h, w = H // P, W // P
    m = mask.double()[:, :, None].repeat(1, 1, P * P * 3).reshape(-1, h, w, P, P, 3).permute(0, 5, 1, 3, 2, 4)
    return m.reshape(-1, 3, H, W).expand(B, 3, H, W)


def _patchify(pred, B, H, W):
    h, w = H // P, W // P
    return pred.reshape(B, 3, h, P, w, P).permute(0, 2, 4, 3, 5, 1).reshape(B, h * w, P * P * 3)


def _decoder_forward(B, H, W, kind, maskB, seggpt, seed):
    """Kernel forward + fp64 reference from the kernel's own bf16 conv output.  Returns everything the checks use."""
    from painter_b200 import ops
    g, c3w, hp, tgts, mask, valid = _decoder_inputs(B, H, W, seed, maskB)
    wf, wd = ops.conv3x3_pack(c3w)
    st = ops.loss_prep(tgts, mask, valid, P)
    c1, patch, num = ops.decoder_head_fwd(g, wf, hp, tgts, mask, valid, P, kind)
    loss, coef = ops.loss_finalize(st, num, seggpt)
    w64 = c3w.bfloat16().double()
    g64 = g.double().permute(0, 3, 1, 2)
    conv = F.conv2d(g64, w64, hp[:64].double(), padding=1)
    S = F.conv2d(g64.abs(), w64.abs(), hp[:64].double().abs(), padding=1)
    assert_close(c1.permute(0, 3, 1, 2), conv, bf16_ulp(conv) + 1e-5 * S, "conv3x3 output c1")
    c1_64 = c1.double().requires_grad_(True)
    pred, mag = _head_from_c1(c1_64, hp)
    assert_close(patch, _patchify(pred.detach(), B, H, W), 1e-5 * _patchify(mag, B, H, W), "patch")
    M = _mask_pixels(mask, B, H, W)
    v = valid.double().clone()
    if not seggpt:   # models_painter.py forward_loss: samples with too little unmasked target are ignored
        mean = torch.tensor(IMNET_MEAN, device=DEV, dtype=torch.float64)[None, :, None, None]
        std = torch.tensor(IMNET_STD, device=DEV, dtype=torch.float64)[None, :, None, None]
        v[((tgts.double() * std + mean) * (1 - M)).sum((1, 2, 3)) < 300] = 0
    wt = M * v
    d = pred - tgts.double()
    rl = (_loss_terms(d, kind) * wt).sum() / (wt.sum() + (0 if seggpt else 1e-2))
    assert abs(loss.item() - rl.item()) <= 1e-4 * abs(rl.item()), (loss.item(), rl.item())
    return dict(g=g, wd=wd, hp=hp, tgts=tgts, mask=mask, valid=valid, c1=c1, coef=coef, c1_64=c1_64, rl=rl, d=d,
                wt=wt, w64=w64)


@pytest.mark.parametrize("B,H,W", DECODER_GEOMETRIES)
def test_decoder_head_broadcast_mask_forward(B, H, W):
    """maskB = 1 (one mask for every sample, the SegGPT form) with the SegGPT loss normalisation; forward only."""
    _decoder_forward(B, H, W, 0, 1, True, seed=W)


@pytest.mark.parametrize("kind", [1, 2, 3])
@pytest.mark.parametrize("B,H,W", DECODER_GEOMETRIES)
def test_decoder_head_loss_kinds_forward_backward(B, H, W, kind):
    from painter_b200 import ops
    r = _decoder_forward(B, H, W, kind, B, False, seed=W + kind)
    gscale = torch.tensor([3.0], device=DEV)
    (r["rl"] * 3.0).backward()
    ref = r["c1_64"].grad
    dc1, dhp = ops.decoder_head_bwd(r["c1"], r["tgts"], r["mask"], r["valid"], r["coef"], gscale, r["hp"], P, kind)
    # l1 / l1l2 have a step in the derivative at d = 0: pixels within rounding distance of it are not comparable
    keep = ((r["d"].abs() > 1e-4) | (r["wt"] == 0)).all(1).permute(0, 1, 2)[..., None]
    floor = 1e-3 * ref.pow(2).mean().sqrt()
    bound = torch.where(keep, bf16_ulp(ref) + floor, torch.full_like(ref, float("inf")))
    assert_close(dc1, ref, bound, "dc1")
    # parameter gradients of LN2D weight / bias, conv1x1 weight / bias (conv3x3 bias: column sums of dc1)
    leaves = [t.detach().clone().requires_grad_(True) for t in (r["hp"][64:128].double(), r["hp"][128:192].double(),
                                                                r["hp"][192:387].double())]
    hp64 = torch.cat([r["hp"][:64].double(), *leaves, r["hp"][387:].double()])
    pred, _ = _head_from_c1(r["c1"].double(), hp64)
    d = pred - r["tgts"].double()
    rl = (_loss_terms(d, kind) * r["wt"]).sum() / (r["wt"].sum() + 1e-2)
    (rl * 3.0).backward()
    for name, got, want in (("LN2D weight", dhp[64:128], leaves[0].grad), ("LN2D bias", dhp[128:192], leaves[1].grad),
                            ("conv1x1", dhp[192:387], leaves[2].grad)):
        assert relmax(got, want) < 1e-3, name
    # conv3x3 gradients from the kernel's own dc1, against torch's convolution gradients in fp64
    dc64 = dc1.double().permute(0, 3, 1, 2)
    g64 = r["g"].double().permute(0, 3, 1, 2)
    dw = ops.conv3x3_wgrad(r["g"], dc1)
    want = torch.nn.grad.conv2d_weight(g64, (64, 64, 3, 3), dc64, padding=1)
    S = torch.nn.grad.conv2d_weight(g64.abs(), (64, 64, 3, 3), dc64.abs(), padding=1)
    assert_close(dw, want, 1e-5 * S, "conv3x3 wgrad")
    h, w = H // P, W // P
    dD = ops.conv3x3_dgrad_unshuffle(dc1, r["wd"], P)
    unshuffle = lambda t: t.permute(0, 2, 3, 1).reshape(B, h, P, w, P, 64).permute(0, 1, 3, 2, 4, 5).reshape(
        B * h * w, P * P * 64)
    want = unshuffle(torch.nn.grad.conv2d_input(g64.shape, r["w64"], dc64, padding=1))
    S = unshuffle(torch.nn.grad.conv2d_input(g64.shape, r["w64"].abs(), dc64.abs(), padding=1))
    assert_close(dD, want, bf16_ulp(want) + 1e-5 * S, "conv3x3 dgrad + unshuffle")


@pytest.mark.parametrize("W", [48, 96])
def test_decoder_refuses_unsupported_widths(W):
    """W = 48 / 96 tile neither into 128-pixel conv tiles nor 64-pixel wgrad tiles: every entry point refuses them
    on the host (before any launch), the head backward included."""
    from painter_b200 import _lib
    L = _lib.lib()
    B, H = 1, 64
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.zeros(B, H, W, 64, dtype=torch.bfloat16, device=DEV)
    wmat = torch.zeros(64, 576, dtype=torch.bfloat16, device=DEV)
    hp = torch.zeros(392, device=DEV)
    tgts, valid = torch.zeros(B, 3, H, W, device=DEV), torch.ones(B, 3, H, W, device=DEV)
    mask = torch.zeros(B, (H // P) * (W // P), dtype=torch.uint8, device=DEV)
    c1 = _nan(B, H, W, 64, dtype=torch.bfloat16)
    patch, num = _nan(B, (H // P) * (W // P), P * P * 3), _nan(B)
    dc1, dhp = _nan(B, H, W, 64, dtype=torch.bfloat16), _nan(392)
    coef, gscale = torch.ones(B, device=DEV), torch.ones(1, device=DEV)
    tok = _nan(B * (H // P) * (W // P), P * P * 64, dtype=torch.bfloat16)
    acc = _nan(640, 64)
    calls = {
        "pk_decoder_head_fwd": lambda: L.pk_decoder_head_fwd(vp(g), vp(wmat), vp(hp), vp(tgts), vp(mask), B, vp(valid),
                                                             vp(c1), vp(patch), vp(num), B, H, W, P, 0, st),
        "pk_decoder_head_bwd": lambda: L.pk_decoder_head_bwd(vp(c1), vp(tgts), vp(mask), B, vp(valid), vp(coef),
                                                             vp(gscale), vp(hp), vp(dc1), vp(dhp), B, H, W, P, 0, st),
        "pk_conv3x3_dgrad_unshuffle": lambda: L.pk_conv3x3_dgrad_unshuffle(vp(dc1), vp(wmat), vp(tok), B, H, W, P, st),
        "pk_conv3x3_wgrad": lambda: L.pk_conv3x3_wgrad(vp(g), vp(dc1), vp(acc), B, H, W, st),
    }
    for name, call in calls.items():
        assert call() != 0, f"{name} accepted W={W}"
        msg = L.pk_last_error().decode()
        assert name in msg and f"{H}x{W}" in msg, msg
    torch.cuda.synchronize()
    for t in (c1, patch, num, dc1, dhp, tok, acc):
        assert bool(torch.isnan(t.float()).all()), "a refused call wrote its output"
