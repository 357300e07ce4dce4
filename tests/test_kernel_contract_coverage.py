"""Host-only view of what test_gpu_kernel_contracts.py's GEMM table reaches: for every case and hook setting the
planner (pk_gemm_plan, the code pk_gemm_bf16 runs; 148 SMs assumed without a device) decides kernel and tile width,
and together the cases must cover every (kernel, BN, epilogue) the planner can produce, with and without bias, and
every tail class of the 256-row tiles of the CTA-pair kernel."""
import pytest

import test_gpu_kernel_contracts as kc

KERNEL_TILES = {0: (64, 128, 256), 1: (128, 256)}    # single CTA, CTA pair


def _reached():
    out = []
    for site, T in kc.gemm_cases():
        M, N, K = site.mnk(T)
        for pair, bn in kc.hooks_for(N):
            with kc.gemm_hooks(pair, bn):
                p = kc.plan(M, N, K, site.kind, site.acc)
            want = kc.expected_kernel(M, N, pair, bn)
            assert want is None or (p["pair"], p["BN"]) == want, (site.name, T, pair, bn, p)
            out.append((site, M, p))
    return out


@pytest.fixture(scope="module")
def reached():
    return _reached()


def test_every_kernel_tile_and_epilogue_is_reached(reached):
    seen = {(p["pair"], p["BN"], s.kind) for s, _, p in reached}
    missing = [(pair, bn, kc.KIND_NAMES[k]) for pair, tiles in KERNEL_TILES.items() for bn in tiles
               for k in kc.KIND_NAMES if (pair, bn, k) not in seen]
    assert not missing, f"(cta_pair, BN, epilogue) never planned: {missing}"


def test_every_epilogue_runs_with_and_without_bias_on_both_kernels(reached):
    seen = {(p["pair"], s.kind, s.bias) for s, _, p in reached}
    missing = [(pair, kc.KIND_NAMES[k], b) for pair in (0, 1) for k in kc.KIND_NAMES for b in (False, True)
               if (pair, k, b) not in seen]
    assert not missing, f"(cta_pair, epilogue, bias) never planned: {missing}"


def test_cta_pair_kernel_sees_every_row_tail(reached):
    """Last 256-row tile full, at most half full (only the first CTA of the pair has rows), more than half full."""
    tails = {"full" if M % 256 == 0 else ("first half" if M % 256 <= 128 else "second half")
             for s, M, p in reached if p["pair"]}
    assert tails == {"full", "first half", "second half"}, tails


def test_default_plan_takes_the_cta_pair_kernel_for_the_model_gemms():
    """With the default heuristics every model-size GEMM (M >= 1568) runs on the CTA-pair kernel, except the
    64-column outputs of the fp32-accurate attention, which only the single-CTA kernel tiles."""
    default = {}
    for site, T in kc.gemm_cases():
        M, N, K = site.mnk(T)
        if min(M, T) < 1568:
            continue
        default[(site.name, T)] = kc.plan(M, N, K, site.kind, site.acc)["pair"]
    single = sorted(k for k, v in default.items() if not v)
    assert all(name == "accurate_pv" for name, _ in single), single
