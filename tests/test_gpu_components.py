"""GPU: connected-component labelling and the component filters (preprocess.label_components / largest_component /
remove_small_components, DESIGN.md section 7c) bit for bit against the scipy oracle of tests/components_oracle.py:
random volumes around the percolation threshold, shapes that are no multiple of any tile, adversarial structures,
batches, dtypes, the full-size bench volumes, CUDA-graph capture and determinism, and the label volumes of
sliding_window_predict."""
import numpy as np
import pytest
import torch

import components_oracle as CC

pytestmark = pytest.mark.gpu

DEV = "cuda"
CONNS = [6, 18, 26]


def _P():
    from ctunet_b200 import preprocess as P
    return P


def _check(mask, conn, min_size=3, filters=True):
    """mask: CPU tensor [D, H, W] or [B, D, H, W].  Labels, counts and both filters must equal the oracle exactly."""
    P = _P()
    m = mask.numpy()
    lab, cnt = P.label_components(mask.to(DEV), conn)
    rl, rc = CC.label(m, conn)
    assert lab.dtype == torch.int32 and lab.shape == mask.shape
    assert cnt.dtype == torch.int64 and cnt.shape == (() if mask.dim() == 3 else (mask.shape[0],))
    assert np.array_equal(lab.cpu().numpy(), rl), (conn, int((lab.cpu().numpy() != rl).sum()))
    assert np.array_equal(cnt.cpu().numpy(), rc)
    if filters:
        big = P.largest_component(mask.to(DEV), conn)
        assert big.dtype == mask.dtype and big.shape == mask.shape
        assert np.array_equal(big.cpu().numpy(), CC.largest(m, conn)), conn
        small = P.remove_small_components(mask.to(DEV), min_size, conn)
        assert np.array_equal(small.cpu().numpy(), CC.remove_small(m, min_size, conn)), conn
    return rc


def _bern(shape, p, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(shape, generator=g) < p).to(torch.uint8)


@pytest.mark.parametrize("conn", CONNS)
@pytest.mark.parametrize("density", [0.05, 0.2, 0.31, 0.5])
def test_random_volumes(density, conn):
    _check(_bern((40, 70, 90), density, 1), conn)           # scalar paths (width not a multiple of 16)
    _check(_bern((32, 64, 96), density, 2), conn, 5)        # 16-byte paths


@pytest.mark.parametrize("conn", CONNS)
@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 37), (3, 5, 7), (17, 33, 65), (33, 130, 129), (64, 64, 64)])
def test_awkward_shapes(shape, conn):
    for p in (0.3, 1.0):
        _check(_bern(shape, p, 3), conn)


def _serpentine(d, h, w):
    """One path through the whole volume: boustrophedon rows in the even planes, one link voxel in the odd ones."""
    m = torch.zeros(d, h, w, dtype=torch.uint8)
    end = None
    for z in range(0, d, 2):
        m[z, 0::2] = 1
        for y in range(1, h, 2):
            m[z, y, w - 1 if (y // 2) % 2 == 0 else 0] = 1
        if end is not None:
            m[z - 1][end] = 1
        yl = (h - 1) // 2 * 2
        end = (yl, w - 1 if (yl // 2) % 2 == 0 else 0)
    return m


@pytest.mark.parametrize("conn", CONNS)
def test_adversarial_structures(conn):
    s = _serpentine(15, 41, 70)
    assert _check(s, conn) == 1
    _check(_serpentine(33, 17, 129), conn)
    _check(_serpentine(16, 16, 64).flip(2).contiguous(), conn)    # the root is found only at the far end of the path
    z, y, x = torch.meshgrid(torch.arange(20), torch.arange(37), torch.arange(48), indexing="ij")
    board = ((x + y + z) % 2 == 1).to(torch.uint8)
    n = _check(board, conn)
    assert n == (int(board.sum()) if conn == 6 else 1)
    diag = torch.zeros(40, 40, 40, dtype=torch.uint8)
    diag[torch.arange(40), torch.arange(40), torch.arange(40)] = 1
    assert _check(diag, conn) == (1 if conn == 26 else 40)
    comb = torch.zeros(37, 45, 100, dtype=torch.uint8)
    comb[0, 0, :] = 1                                              # back bar
    comb[0, :, 0::3] = 1                                           # teeth along y from the bar, across 8-row tiles
    comb[:, 2::5, 1::3] = 1                                        # free pillars along z, across 8-plane tiles
    comb[:, 44, 31:34] = 1                                         # a wall across the 32-column tile boundary
    _check(comb, conn)
    _check(torch.ones(19, 21, 40, dtype=torch.uint8), conn)
    assert _check(torch.zeros(19, 21, 40, dtype=torch.uint8), conn) == 0
    for shape in ((9, 10, 11), (33, 130, 129)):
        corners = torch.zeros(shape, dtype=torch.uint8)
        corners[0::shape[0] - 1, 0::shape[1] - 1, 0::shape[2] - 1] = 1
        assert _check(corners, conn) == 8


@pytest.mark.parametrize("conn", CONNS)
def test_batches_equal_separate_volumes(conn):
    P = _P()
    m = _bern((3, 20, 30, 48), 0.3, 4)
    m[0, -1] = 1                                                   # last plane of volume 0 and first of volume 1 full:
    m[1, 0] = 1                                                    # adjacent in memory, never joined
    rc = _check(m, conn)
    lab, cnt = P.label_components(m.to(DEV), conn)
    for b in range(3):
        lb, cb = P.label_components(m[b].to(DEV), conn)
        assert torch.equal(lab[b], lb) and int(cnt[b]) == int(cb) == int(rc[b])
        assert torch.equal(P.largest_component(m.to(DEV), conn)[b], P.largest_component(m[b].to(DEV), conn))
    _check(_bern((5, 7, 9, 11), 0.4, 5), conn)
    _check(torch.zeros(2, 4, 4, 16, dtype=torch.uint8), conn)


@pytest.mark.parametrize("conn", CONNS)
def test_dtypes_give_identical_labels(conn):
    P = _P()
    g = torch.Generator().manual_seed(6)
    cls = torch.randint(0, 3, (24, 40, 64), generator=g) * (torch.rand(24, 40, 64, generator=g) < 0.4)
    f32 = cls.float()                                              # class values {0, 1, 2}
    ref = _check(f32, conn)
    for t in (cls.to(torch.uint8), cls != 0, f32[:, :, :61].contiguous()):
        _check(t, conn)
    labs = [P.label_components(t.to(DEV), conn)[0] for t in (f32, cls.to(torch.uint8), cls != 0)]
    assert torch.equal(labs[0], labs[1]) and torch.equal(labs[0], labs[2])
    big = P.largest_component(f32.to(DEV), conn).cpu()
    keep = big != 0
    assert big.dtype == torch.float32 and torch.equal(big[keep], f32[keep])      # kept voxels keep their class
    assert set(big.unique().tolist()) <= {0.0, 1.0, 2.0} and int(ref) >= 1
    assert P.largest_component((cls != 0).to(DEV), conn).dtype == torch.bool


@pytest.mark.parametrize("shape", [(256, 512, 512), (224, 512, 512)])
def test_full_size_bench_volumes(shape):
    from ctunet_b200 import synthetic
    P = _P()
    mask = P.hu_threshold(synthetic.head_ct_hu(shape, seed=0, device=DEV), 300)
    m = mask.cpu().numpy()
    for conn in (6, 26):
        lab, cnt = P.label_components(mask, conn)
        rl, rc = CC.label(m, conn)
        assert int(cnt) == int(rc) and int(rc) > 1000
        assert np.array_equal(lab.cpu().numpy(), rl)
        big = P.largest_component(mask, conn).cpu().numpy()
        assert np.array_equal(big, CC.largest(m, conn))
        assert big.sum() > 10 ** 6                                 # the skull


def test_graph_capture_and_determinism():
    P = _P()
    a = _bern((40, 64, 96), 0.31, 7).to(DEV)
    b = _bern((40, 64, 96), 0.31, 8).to(DEV)
    static = a.clone()
    P.largest_component(static, 26)
    P.label_components(static, 26)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        big = P.largest_component(static, 26)
        lab, cnt = P.label_components(static, 26)
    static.copy_(b)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(big, P.largest_component(b, 26))
    assert torch.equal(lab, P.label_components(b, 26)[0]) and torch.equal(cnt, P.label_components(b, 26)[1])
    assert np.array_equal(big.cpu().numpy(), CC.largest(b.cpu().numpy(), 26))
    big_a = P.largest_component(a, 6)
    assert torch.equal(big_a, P.largest_component(a, 6))          # two runs, bit-identical
    assert torch.equal(P.label_components(a, 18)[0], P.label_components(a, 18)[0])


def test_composes_with_sliding_window_predict():
    import ctunet_b200 as C
    P = _P()
    torch.manual_seed(0)
    net = C.UNetSP().to(DEV).eval()
    vol = (torch.rand(2, 24, 56, 70, generator=torch.Generator().manual_seed(9)) > 0.7).float().to(DEV)
    labels = P.sliding_window_predict(net, vol, patch=32, overlap=0.5)
    flap = labels[1]
    assert flap.dtype == torch.float32 and flap.shape == (24, 56, 70)
    f = flap.cpu().numpy()
    for conn in CONNS:
        assert np.array_equal(P.largest_component(flap, conn).cpu().numpy(), CC.largest(f, conn))
        assert np.array_equal(P.remove_small_components(flap, 10, conn).cpu().numpy(), CC.remove_small(f, 10, conn))


def test_gpu_argument_errors():
    P = _P()
    m = torch.zeros(4, 4, 4, dtype=torch.uint8, device=DEV)
    with pytest.raises(TypeError):
        P.label_components(m.to(torch.int32))
    with pytest.raises(ValueError):
        P.label_components(m, 10)
    with pytest.raises(ValueError):
        P.remove_small_components(m, -2)
    lab, cnt = P.label_components(torch.zeros(0, 4, 4, dtype=torch.uint8, device=DEV))
    assert lab.shape == (0, 4, 4) and int(cnt) == 0
