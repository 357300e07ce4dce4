"""Worst error of the GEMM-epilogue GELU (EPI_GELU) and GELU' (EPI_DGELU) over every finite bf16 input |z| <= 12, per
range of z, on both GEMM kernels: in bf16 ulps of the true value and as a fraction of the bounds the kernel tests
hold it to (GELU: 1 ulp + 2^-15; GELU': 1 ulp + |acc| 2^-13).  PK_LIB selects a tuning build.
Usage (GPU box): python scripts/gelu_epilogue_error.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
import test_gpu_kernel_contracts as kc  # noqa: E402
from painter_b200 import ops  # noqa: E402

zs = kc.all_bf16_upto(12.0)
a, b, bt, n = kc._identity_gemm_operands(zs, 0.0)
a512 = torch.eye(512, device="cuda").bfloat16()
for pair, bn in kc.GELU_HOOKS:
    name = f"{'cta-pair' if kc.expected_kernel(512, 128, pair, bn)[0] else 'single-cta'} BN={bn}"
    with kc.gemm_hooks(pair, bn):
        z, h = ops.gemm(a, b, kind=kc.EPI_GELU)
    zf = z.double().flatten()[:n]
    want = kc.gelu64(zf)
    print(f"GELU  {name:20s}", kc._fmt(kc.gelu_errors(zf, h.flatten()[:n], want, torch.full_like(want, 2.0 ** -15))))
    for c in (1.0, -3.0, 0.375, 96.0):
        bc = torch.full((128, 512), c, device="cuda").bfloat16()
        with kc.gemm_hooks(pair, bn):
            d = ops.gemm(a512, bc, kind=kc.EPI_DGELU, aux=bt)
        want = c * kc.gelu_grad64(zf)
        rows = kc.gelu_errors(zf, d.flatten()[:n], want, torch.full_like(want, abs(c) * 2.0 ** -13))
        print(f"GELU' {name:20s} acc={c:g}:", kc._fmt(rows))
