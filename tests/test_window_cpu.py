"""CPU: the window grid, weight and normaliser tables of overlapping sliding-window inference
(preprocess.window_origins / window_weights / window_normaliser / window_grid) against the independent oracle of
tests/window_oracle.py, and the argument checks that need no device."""
import numpy as np
import pytest
import torch

from ctunet_b200 import preprocess as P
import window_oracle as W

OVERLAPS = [0.0, 0.25, 0.5, 0.75]
PATCHES = [4, 16, 32, 128]


def _sizes(p):
    return sorted({1, 3, p - 1, p, p + 1, 2 * p - 3, 2 * p, 2 * p + 1, 3 * p + 5, 4 * p} - {0})


@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("patch", PATCHES)
def test_origins_match_oracle_and_cover_every_voxel(patch, overlap):
    for s in _sizes(patch):
        got = P.window_origins(s, patch, overlap)
        assert got == W.axis_origins(s, patch, overlap), (s, patch, overlap)
        assert all(0 <= o <= max(s - patch, 0) for o in got)
        assert got == sorted(set(got)) and got[0] == 0
        cover = np.zeros(s, dtype=np.int64)
        for o in got:
            cover[o:o + patch] += 1
        assert cover.min() >= 1, (s, patch, overlap)
        if s > patch:
            assert got[-1] == s - patch                      # the last window ends at the border
            step = max(1, int(np.floor(patch * (1 - overlap))))
            assert len(got) == -(-(s - patch) // step) + 1


def test_worked_examples():
    n = lambda shape, ov: int(np.prod([len(P.window_origins(s, 128, ov)) for s in shape]))
    assert n((224, 512, 512), 0.0) == 32 and n((224, 512, 512), 0.5) == 147
    assert n((256, 512, 512), 0.0) == 32 and n((256, 512, 512), 0.5) == 147
    assert P.window_origins(512, 128, 0.0) == [0, 128, 256, 384]        # the grid sliding_window_argmax uses
    assert P.window_origins(224, 128, 0.0) == [0, 96]


@pytest.mark.parametrize("patch", PATCHES + [7, 96])
@pytest.mark.parametrize("sigma_scale", [0.05, 0.125, 0.5])
def test_weights_match_oracle(patch, sigma_scale):
    g = P.window_weights(patch, "gaussian", sigma_scale)
    assert g.dtype == np.float64 and g.shape == (patch,)
    np.testing.assert_allclose(g, W.axis_weights(patch, "gaussian", sigma_scale), rtol=1e-15, atol=0)
    assert np.array_equal(g, g[::-1])                                   # symmetric
    assert g.max() == 1.0 and g.min() >= 2.0 ** -6
    if sigma_scale <= 0.125 and patch >= 16:
        assert g.min() == 2.0 ** -6                                     # the floor is reached at the window edges
    assert np.array_equal(P.window_weights(patch, "constant"), np.ones(patch))


@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("blend", ["constant", "gaussian"])
def test_normaliser_matches_oracle(overlap, blend):
    for patch in (16, 32):
        wt = P.window_weights(patch, blend)
        for s in _sizes(patch):
            org = P.window_origins(s, patch, overlap)
            got = P.window_normaliser(s, patch, org, wt)
            np.testing.assert_allclose(got, W.axis_normaliser(s, patch, org, list(wt)), rtol=1e-14)
            assert got.min() >= 2.0 ** -6                               # every voxel has weight


def test_grid_and_overflow_guard():
    axes = P.window_grid((24, 56, 70), 32, 0.5)
    assert axes == [[0], [0, 16, 24], [0, 16, 32, 38]]
    P.window_grid((512, 512, 512), 128, 0.99)                           # step 1 at p = 128: 2^21 windows cover a voxel
    with pytest.raises(OverflowError):
        P.window_grid((400, 400, 400), 200, 0.999)                      # step 1 at p = 200: 8e6 windows > 2^22
    P.window_grid((170, 170, 170), 162, 0.999)                          # only 9 origins per axis
    with pytest.raises(OverflowError):
        P.window_grid((400, 400, 400), 162, 0.999)                      # 162^3 > 2^22


def test_sliding_window_predict_rejects_cpu_and_bad_arguments():
    import ctunet_b200 as C
    net = C.UNetSP()
    with pytest.raises(RuntimeError):
        P.sliding_window_predict(net, torch.zeros(2, 32, 32, 32), patch=32)
    with pytest.raises(ValueError):
        P.window_weights(32, "cosine")
