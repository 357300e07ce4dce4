"""GPU data-path kernels (SURVEY §8 f.4) against the unmodified reference: the block-mask generator keeps the
reference's invariants and statistics (its random source differs, so parity is distributional), the `valid` maps are
bit-identical to PairDataset.__getitem__ (driven on temporary image files).  The reference side is stored in
tests/golden/ref_datapath.pt (`python -m oracle.make_golden datapath`)."""
import numpy as np
import pytest
import torch

from oracle.make_golden import to_normalised

from _common import load_golden

pytestmark = pytest.mark.gpu


def _blockiness(m):
    m = m.astype(np.float64)
    return ((m[:, 1:, :] == m[:, :-1, :]).mean() + (m[:, :, 1:] == m[:, :, :-1]).mean()) / 2


def test_block_masks_invariants_and_statistics_vs_reference_generator():
    from painter_b200.data_gpu import DeviceMaskingGenerator
    ref = load_golden("ref_datapath.pt")["masks"]
    h, w, target = 56, 28, 784
    ours = DeviceMaskingGenerator((h, w), num_masking_patches=target, max_num_patches=392, min_num_patches=16)
    n = 1024
    mo = torch.cat([ours(256, seed=100 + k) for k in range(n // 256)]).cpu().numpy()
    assert mo.shape == (n, h, w) and set(np.unique(mo)) <= {0, 1}
    assert (mo.reshape(n, -1).sum(1) == target).all()                                  # exact count, every sample
    assert len({m.tobytes() for m in mo}) == n                                         # all different
    # same structure as 1024 draws of the reference generator: block-iness (neighbour agreement) and the spatial
    # masking profile
    assert abs(_blockiness(mo) - ref["blockiness"]) < 0.01, (_blockiness(mo), ref["blockiness"])
    assert np.abs(mo.mean(0) - ref["mean_map"].numpy()).max() < 0.08
    assert np.abs(mo.mean((0, 2)) - ref["row_marginal"].numpy()).max() < 0.03          # per-row marginal
    assert np.abs(mo.mean((0, 1)) - ref["col_marginal"].numpy()).max() < 0.03          # per-column marginal
    # the half-mask alternative (pairdataset.py:183-186)
    half = DeviceMaskingGenerator((h, w), target, max_num_patches=392, min_num_patches=16, half_mask_ratio=1.0)(4, 7)
    want = torch.zeros(h, w, dtype=torch.int32)
    want[h // 2:] = 1
    assert all(torch.equal(m.cpu(), want) for m in half)
    mix = DeviceMaskingGenerator((h, w), target, max_num_patches=392, min_num_patches=16, half_mask_ratio=0.1)(2000, 3)
    frac = float(np.mean([torch.equal(m, want.cuda()) for m in mix]))
    assert 0.06 < frac < 0.14, frac


def test_valid_maps_bit_identical_to_pairdataset():
    """PairDataset.__getitem__ on the 12 image pairs of oracle.make_golden.datapath_pairs (all six task types, black
    regions, an almost empty pose target, an empty instance target): its targets, rebuilt from the stored pixels, give
    painter_b200's valid maps bit for bit equal to the ones it returned."""
    from painter_b200.data_gpu import combine_pairs, valid_maps
    ref = load_golden("ref_datapath.pt")
    tg = torch.stack([to_normalised(u) for u in ref["targets_u8"]])
    assert tuple(tg.shape[1:]) == (3, 128, 64)
    ours = valid_maps(tg.cuda().contiguous(), ref["types"])
    vd = ref["valid"].float()
    for i, v in enumerate(vd):
        assert torch.equal(ours[i].cpu(), v), (ref["types"][i], (ours[i].cpu() != v).sum())
    assert {float(x) for x in vd.unique()} == {0.0, 1.0, 10.0}       # all three branches were exercised
    c = ref["combine"]
    assert torch.equal(combine_pairs(c["a"], c["b"])[0], c["out"])
