"""GPU: utilities.surface_metrics (DESIGN.md section 7d) against the scipy / numpy oracle of tests/surface_oracle.py.

Unit spacing: dice, hausdorff, hausdorff_percentile and surface_dice bit for bit, assd to relative 1e-12 (numpy sums
pairwise in another order).  With spacing: distances to relative 1e-12, counts exact unless the tolerance lies within
1e-9 of an attainable distance.  Smooth random blob pairs on tile-aligned and unaligned shapes, single slices and rows,
batches, every dtype pair, percentiles and tolerances that hit attainable distances, degenerate cases, agreement with
utilities.hausdorff, the full-size head CT, and CUDA-graph replay."""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage

import surface_oracle as SO

pytestmark = pytest.mark.gpu

DEV = "cuda"
PERCENTILES = [0.0, 50.0, 95.0, 99.5, 100.0]
TOLERANCES = [0.0, 1.0, math.sqrt(2.0), 2.2]
DISTANCES = ("hausdorff", "hausdorff_percentile", "assd")


def _sm(*args, **kw):
    from ctunet_b200.utilities import surface_metrics
    return surface_metrics(*args, **kw)


def _blob_pair(shape, seed, sigma=2.0):
    """Two overlapping smooth random blobs (uint8, CPU): Gaussian-smoothed noise thresholded at its median, the second
    from the same field plus an independent perturbation so that the surfaces are near but not equal."""
    rng = np.random.default_rng(seed)
    base = ndimage.gaussian_filter(rng.standard_normal(shape), sigma, mode="wrap")
    pert = ndimage.gaussian_filter(rng.standard_normal(shape), sigma, mode="wrap")
    a = base > np.median(base)
    b = base + 0.6 * pert * base.std() / max(pert.std(), 1e-12) > np.median(base)
    return torch.from_numpy(a.astype(np.uint8)), torch.from_numpy(b.astype(np.uint8))


def _as(t, dtype):
    return t.to(dtype).to(DEV)


def _check_exact(got, ref):
    """Unit spacing: bit-equal, assd to 1e-12."""
    for k in SO.KEYS:
        g = got[k].cpu().numpy()
        assert got[k].dtype == torch.float64 and g.shape == np.shape(ref[k]), k
        if k == "assd":
            finite = np.isfinite(ref[k])
            assert np.array_equal(np.isfinite(g), finite) and np.array_equal(np.isnan(g), np.isnan(ref[k])), k
            assert np.allclose(g[finite], np.asarray(ref[k])[finite], rtol=1e-12, atol=0), (k, g, ref[k])
            assert np.array_equal(g[~finite], np.asarray(ref[k])[~finite], equal_nan=True), k
        else:
            assert np.array_equal(g, ref[k], equal_nan=True), (k, g.tolist(), np.asarray(ref[k]).tolist())


def _attainable(p, t, spacing):
    """Every distance value of both directed sets (for the 'not near an attainable distance' test)."""
    vols_p, vols_t = (p[None], t[None]) if p.ndim == 3 else (p, t)
    out = []
    for a, b in zip(vols_p, vols_t):
        if a.any() and b.any():
            ea, eb = SO.edges(a), SO.edges(b)
            out += [SO.directed(ea, eb, spacing), SO.directed(eb, ea, spacing)]
    return np.concatenate(out) if out else np.zeros(0)


@pytest.mark.parametrize("shape", [(32, 32, 32), (24, 40, 56), (17, 33, 65), (1, 30, 40), (1, 1, 70)])
def test_unit_spacing_matches_oracle(shape):
    p, t = _blob_pair(shape, seed=sum(shape))
    for q in PERCENTILES:
        for tol in TOLERANCES:
            got = _sm(_as(p, torch.uint8), _as(t, torch.uint8), percentile=q, tolerance=tol)
            _check_exact(got, SO.surface_metrics(p.numpy(), t.numpy(), percentile=q, tolerance=tol))


def test_batches_of_three():
    pairs = [_blob_pair((24, 40, 56), seed=s) for s in (1, 2, 3)]
    p = torch.stack([a for a, _ in pairs])
    t = torch.stack([b for _, b in pairs])
    t[1] = torch.roll(t[1], 3, dims=2)
    for q, tol in ((95.0, 1.0), (50.0, math.sqrt(2.0))):
        got = _sm(_as(p, torch.uint8), _as(t, torch.uint8), percentile=q, tolerance=tol)
        assert got["dice"].shape == (3,)
        _check_exact(got, SO.surface_metrics(p.numpy(), t.numpy(), percentile=q, tolerance=tol))


@pytest.mark.parametrize("pdt", [torch.uint8, torch.bool, torch.float32])
@pytest.mark.parametrize("tdt", [torch.uint8, torch.bool, torch.float32])
def test_every_dtype_pair(pdt, tdt):
    p, t = _blob_pair((17, 33, 65), seed=11)
    pv = p.to(pdt)
    tv = t.to(tdt)
    if tdt == torch.float32:
        # any non-zero value is foreground; a local generator leaves torch's global RNG state to the tests that follow
        u = torch.rand(tv.shape, generator=torch.Generator().manual_seed(12))
        tv = tv * torch.where(u < 0.5, -3.5, 0.25)
    got = _sm(pv.to(DEV), tv.to(DEV), percentile=99.5, tolerance=2.2)
    _check_exact(got, SO.surface_metrics(p.numpy(), t.numpy(), percentile=99.5, tolerance=2.2))


@pytest.mark.parametrize("spacing", [(1.5, 0.7, 0.7), (2.0, 1.0, 1.0), (0.5, 0.5, 3.0)])
@pytest.mark.parametrize("shape", [(24, 40, 56), (17, 33, 65)])
def test_with_spacing(spacing, shape):
    p, t = _blob_pair(shape, seed=5)
    p = torch.stack([p, t, torch.roll(p, 2, dims=1)])
    t = torch.stack([t, torch.roll(t, 1, dims=0), p[0]])
    pn, tn = p.numpy(), t.numpy()
    dists = _attainable(pn, tn, spacing)
    for q in PERCENTILES:
        for tol in TOLERANCES + [1.4, 2.1]:
            got = _sm(_as(p, torch.uint8), _as(t, torch.float32), spacing=spacing, percentile=q, tolerance=tol)
            ref = SO.surface_metrics(pn, tn, spacing=spacing, percentile=q, tolerance=tol)
            assert np.array_equal(got["dice"].cpu().numpy(), ref["dice"])
            for k in DISTANCES:
                assert np.allclose(got[k].cpu().numpy(), ref[k], rtol=1e-12, atol=0), (k, q, spacing)
            if np.abs(dists - tol).min() > 1e-9:
                assert np.array_equal(got["surface_dice"].cpu().numpy(), ref["surface_dice"]), (tol, spacing)


def test_edge_cases():
    shape = (9, 10, 11)
    z = torch.zeros(shape, dtype=torch.uint8)
    one = z.clone()
    one[4, 5, 6] = 1
    other = z.clone()
    other[0, 9, 10] = 1
    full = torch.ones(shape, dtype=torch.uint8)
    corner = z.clone()
    corner[:3, :4, :5] = 1
    border = z.clone()
    border[0] = 1
    border[:, :, -1] = 1
    frame = full.clone()
    frame[1:-1, 1:-1, 1:-1] = 0
    cases = [(z, z), (z, one), (one, z), (one, one), (one, other), (full, corner), (corner, full), (full, full),
             (border, frame), (frame, corner), (full, z)]
    for sp in (None, (2.0, 1.0, 0.5)):
        for a, b in cases:
            for q, tol in ((95.0, 1.0), (0.0, 0.0), (100.0, 2.2)):
                got = _sm(_as(a, torch.uint8), _as(b, torch.bool), spacing=sp, percentile=q, tolerance=tol)
                ref = SO.surface_metrics(a.numpy(), b.numpy(), spacing=sp, percentile=q, tolerance=tol)
                for k in SO.KEYS:
                    g = float(got[k])
                    exact = k != "assd" if sp is None else k not in DISTANCES
                    if exact or not math.isfinite(ref[k]):
                        assert g == ref[k] or (math.isnan(g) and math.isnan(ref[k])), (k, g, ref[k])
                    else:
                        assert g == pytest.approx(float(ref[k]), rel=1e-12, abs=0), (k, g, ref[k])
    r = _sm(_as(z, torch.uint8), _as(z, torch.uint8))
    assert all(math.isnan(float(r[k])) for k in SO.KEYS) and r["dice"].dim() == 0


def test_percentile_100_and_utilities_hausdorff():
    from ctunet_b200.utilities import hausdorff
    for shape, seed in (((32, 32, 32), 1), ((17, 33, 65), 2), ((1, 30, 40), 3)):
        p, t = _blob_pair(shape, seed)
        got = _sm(_as(p, torch.uint8), _as(t, torch.uint8), percentile=100.0)
        assert torch.equal(got["hausdorff_percentile"], got["hausdorff"])
        onehot = lambda m: torch.stack([1 - m.float(), m.float()])[None].to(DEV)    # noqa: E731
        assert float(got["hausdorff"]) == float(hausdorff(onehot(p), onehot(t)))
        sp = _sm(_as(p, torch.uint8), _as(t, torch.uint8), spacing=(1.5, 0.7, 0.7), percentile=100.0)
        assert torch.equal(sp["hausdorff_percentile"], sp["hausdorff"])


def _skull_pair(shape):
    """The largest component of the thresholded head CT (the skull), and a copy shifted by (2, -3, 1) voxels with
    about 700 added one-voxel islands."""
    from ctunet_b200 import preprocess as P
    from ctunet_b200 import synthetic
    skull = P.largest_component(P.hu_threshold(synthetic.head_ct_hu(shape, seed=0, device=DEV), 300))
    moved = torch.zeros_like(skull)
    moved[2:, :-3, 1:] = skull[:-2, 3:, :-1]
    g = torch.Generator(device=DEV).manual_seed(1)
    moved[torch.rand(shape, device=DEV, generator=g) < 1e-5] = 1
    return skull, moved


def test_full_size_skull_pair():
    p, t = _skull_pair((256, 512, 512))
    pn, tn = p.cpu().numpy(), t.cpu().numpy()
    got = _sm(p, t, percentile=95.0, tolerance=1.0)
    _check_exact(got, SO.surface_metrics(pn, tn, percentile=95.0, tolerance=1.0))
    sp = (1.25, 0.5, 0.5)
    got = _sm(p, t, spacing=sp, percentile=95.0, tolerance=1.3)
    ref = SO.surface_metrics(pn, tn, spacing=sp, percentile=95.0, tolerance=1.3)
    assert float(got["dice"]) == ref["dice"] and float(got["surface_dice"]) == ref["surface_dice"]
    for k in DISTANCES:
        assert float(got[k]) == pytest.approx(float(ref[k]), rel=1e-12, abs=0), k


def test_graph_replay_and_repeat_calls():
    p, t = _blob_pair((24, 40, 56), seed=21)
    p2, t2 = _blob_pair((24, 40, 56), seed=22)
    for sp in (None, (1.5, 0.7, 0.7)):
        sp_, st_ = _as(p, torch.uint8), _as(t, torch.float32)
        first = _sm(sp_, st_, spacing=sp, percentile=99.5, tolerance=1.0)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cap = _sm(sp_, st_, spacing=sp, percentile=99.5, tolerance=1.0)
        for _ in range(2):
            g.replay()
            torch.cuda.synchronize()
            for k in SO.KEYS:
                assert torch.equal(cap[k], first[k]), k
        again = _sm(sp_, st_, spacing=sp, percentile=99.5, tolerance=1.0)
        for k in SO.KEYS:
            assert torch.equal(again[k], first[k]), k
        sp_.copy_(_as(p2, torch.uint8))                     # the captured graph reads the new inputs
        st_.copy_(_as(t2, torch.float32))
        g.replay()
        ref = _sm(_as(p2, torch.uint8), _as(t2, torch.uint8), spacing=sp, percentile=99.5, tolerance=1.0)
        torch.cuda.synchronize()
        for k in SO.KEYS:
            assert torch.equal(cap[k], ref[k]), k
