"""CPU: the surface-metrics oracle (tests/surface_oracle.py) on hand-computed cases and its degenerate rules, and the
argument checks of utilities.surface_metrics that need no device."""
import math

import numpy as np
import pytest
import torch

import surface_oracle as SO
from ctunet_b200.utilities import surface_metrics


def _voxels(shape, *points):
    m = np.zeros(shape, np.uint8)
    for p in points:
        m[p] = 1
    return m


def test_single_voxels_offset_by_3_4_0_are_5_apart():
    p = _voxels((8, 8, 8), (1, 1, 2))
    t = _voxels((8, 8, 8), (4, 5, 2))
    r = SO.surface_metrics(p, t, percentile=50.0, tolerance=5.0)
    assert r["dice"] == 0.0
    for k in ("hausdorff", "hausdorff_percentile", "assd"):
        assert r[k] == 5.0, k
    assert r["surface_dice"] == 1.0                         # 5 <= 5
    assert SO.surface_metrics(p, t, tolerance=4.999)["surface_dice"] == 0.0


def test_spacing_scales_a_one_slice_offset():
    p = np.zeros((6, 5, 5), np.uint8)
    t = np.zeros((6, 5, 5), np.uint8)
    p[2] = 1
    t[3] = 1                                                # every edge voxel is one slice from the other surface
    r = SO.surface_metrics(p, t, spacing=(2.0, 1.0, 1.0), tolerance=1.5)
    assert r["hausdorff"] == r["hausdorff_percentile"] == r["assd"] == 2.0
    assert r["surface_dice"] == 0.0 and r["dice"] == 0.0
    assert SO.surface_metrics(p, t)["hausdorff"] == 1.0     # voxel units


def test_percentile_is_sort_and_interpolate():
    rng = np.random.default_rng(0)
    vals = np.sqrt(rng.integers(0, 200, size=57).astype(np.float64))
    for q in (0.0, 12.5, 50.0, 95.0, 99.5, 100.0, 100 / 3):
        assert np.percentile(vals, q) == SO.linear_percentile(vals, q), q
    assert SO.linear_percentile([7.0], 40.0) == 7.0


def test_directed_distances_on_a_hand_built_pair():
    p = np.zeros((1, 1, 9), np.uint8)
    t = np.zeros((1, 1, 9), np.uint8)
    p[0, 0, 0:3] = 1                                        # edges 0, 1, 2 (a row: nothing is interior)
    t[0, 0, 6] = 1
    d = SO.directed(SO.edges(p), SO.edges(t))
    assert d.tolist() == [6.0, 5.0, 4.0]
    r = SO.surface_metrics(p, t, percentile=50.0, tolerance=4.0)
    # d(P->T) = {6, 5, 4}, d(T->P) = {4}
    assert r["hausdorff"] == 6.0 and r["hausdorff_percentile"] == 5.0 and r["assd"] == 19 / 4
    assert r["surface_dice"] == 2 / 4 and r["dice"] == 0.0


def test_interior_voxels_are_not_edges():
    m = np.zeros((5, 5, 5), np.uint8)
    m[1:4, 1:4, 1:4] = 1
    e = SO.edges(m)
    assert e.sum() == 26 and not e[2, 2, 2]
    full = np.ones((3, 3, 3), np.uint8)
    assert SO.edges(full).sum() == 26                       # outside the volume counts as background


def test_degenerate_rules():
    z = np.zeros((4, 4, 4), np.float32)
    one = z.copy()
    one[1, 2, 3] = 1
    r = SO.surface_metrics(z, z)
    assert all(math.isnan(r[k]) for k in SO.KEYS)
    for a, b in ((one, z), (z, one)):
        r = SO.surface_metrics(a, b)
        assert r["dice"] == 0.0 and r["surface_dice"] == 0.0
        assert r["hausdorff"] == r["hausdorff_percentile"] == r["assd"] == math.inf
    r = SO.surface_metrics(one, one, percentile=0.0, tolerance=0.0)
    assert r["dice"] == 1.0 and r["surface_dice"] == 1.0 and r["hausdorff"] == 0.0 and r["assd"] == 0.0


def test_batches_are_scored_per_volume():
    p = np.zeros((3, 4, 4, 4), np.uint8)
    t = np.zeros((3, 4, 4, 4), np.uint8)
    p[1, 0, 0, 0] = 1
    t[1, 0, 0, 3] = 1
    p[2, 1, 1, 1] = t[2, 1, 1, 1] = 1
    r = SO.surface_metrics(p, t)
    assert r["hausdorff"].shape == (3,) and r["hausdorff"].dtype == np.float64
    assert math.isnan(r["hausdorff"][0]) and r["hausdorff"][1] == 3.0 and r["hausdorff"][2] == 0.0
    for k in SO.KEYS:
        for i in range(3):
            assert np.array_equal(r[k][i], SO.surface_metrics(p[i], t[i])[k], equal_nan=True), (k, i)


def test_argument_errors_without_a_device():
    m = torch.zeros(4, 4, 4, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        surface_metrics(m, m)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        surface_metrics(m.numpy(), m)
    bad_values = [
        ((torch.zeros(4, 4, dtype=torch.uint8),) * 2, {}),                                      # rank
        ((torch.zeros(1, 1, 4, 4, 4, dtype=torch.uint8),) * 2, {}),
        ((m, torch.zeros(4, 4, 5, dtype=torch.uint8)), {}),                                     # shape mismatch
        ((torch.zeros(2, 4, 4, 4, dtype=torch.uint8), m), {}),
        ((torch.zeros(1, dtype=torch.uint8).expand(4, 4, 1025),) * 2, {}),                      # axis > 1024
        ((torch.zeros(4, 0, 4, dtype=torch.uint8),) * 2, {}),                                   # empty axis
        ((m, m), {"spacing": (1.0, 1.0)}),
        ((m, m), {"spacing": (1.0, 0.0, 1.0)}),
        ((m, m), {"spacing": (1.0, -2.0, 1.0)}),
        ((m, m), {"spacing": (1.0, math.inf, 1.0)}),
        ((m, m), {"spacing": (1.0, math.nan, 1.0)}),
        ((m, m), {"spacing": 1.0}),
        ((m, m), {"spacing": ("1", 1.0, 1.0)}),
        ((m, m), {"percentile": -0.1}),
        ((m, m), {"percentile": 100.5}),
        ((m, m), {"percentile": math.nan}),
        ((m, m), {"percentile": "95"}),
        ((m, m), {"tolerance": -1.0}),
        ((m, m), {"tolerance": math.nan}),
    ]
    for args, kw in bad_values:
        with pytest.raises(ValueError):
            surface_metrics(*args, **kw)
    for dt in (torch.int16, torch.int32, torch.float64, torch.float16):
        with pytest.raises(TypeError):
            surface_metrics(m.to(dt), m)
        with pytest.raises(TypeError):
            surface_metrics(m, m.to(dt))
    for dt in (torch.uint8, torch.bool, torch.float32):    # accepted dtypes get as far as the device check
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            surface_metrics(m.to(dt), m.float(), spacing=[0.5, 0.5, 3], percentile=100, tolerance=0)
