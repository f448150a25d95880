"""CPU: the connected-component oracle (tests/components_oracle.py) on hand-made cases, the raster-order numbering it
asserts on random volumes, and the argument checks of preprocess.label_components / largest_component /
remove_small_components that need no device."""
import numpy as np
import pytest
import torch

import components_oracle as CC
from ctunet_b200 import preprocess as P

CONNS = [6, 18, 26]


def _first_voxel_order(labels, n):
    """Labels in the raster order of their first voxel."""
    flat = labels.ravel()
    _, first = np.unique(flat, return_index=True)
    seen = flat[np.sort(first)]
    return [int(v) for v in seen if v != 0] == list(range(1, n + 1))


@pytest.mark.parametrize("conn", CONNS)
def test_numbering_is_first_voxel_raster_order(conn):
    rng = np.random.default_rng(conn)
    for density in (0.05, 0.2, 0.31, 0.5):
        m = (rng.random((9, 13, 17)) < density).astype(np.uint8)
        lab, n = CC.label(m, conn)
        assert lab.dtype == np.int32 and lab.shape == m.shape and int(n) == lab.max()
        assert _first_voxel_order(lab, int(n)), (conn, density)


def test_empty_and_full_volumes():
    for conn in CONNS:
        lab, n = CC.label(np.zeros((4, 5, 6), np.uint8), conn)
        assert n == 0 and not lab.any()
        assert not CC.largest(np.zeros((4, 5, 6), np.uint8), conn).any()
        full = np.ones((4, 5, 6), np.uint8)
        lab, n = CC.label(full, conn)
        assert n == 1 and (lab == 1).all()
        assert np.array_equal(CC.largest(full, conn), full)
        assert np.array_equal(CC.remove_small(full, 120, conn), full)
        assert not CC.remove_small(full, 121, conn).any()


def test_parity_checkerboard():
    z, y, x = np.indices((6, 7, 8))
    m = ((x + y + z) % 2 == 1).astype(np.uint8)
    lab, n = CC.label(m, 6)
    assert n == m.sum()                                    # every voxel isolated under face connectivity
    for conn in (18, 26):
        lab, n = CC.label(m, conn)
        assert n == 1                                      # edge neighbours join them all
    out = CC.largest(m, 6)                                 # all size 1: the first voxel in raster order wins
    assert out.sum() == 1 and out[0, 0, 1] == 1


def test_space_diagonal_connects_only_under_26():
    m = np.zeros((5, 5, 5), np.uint8)
    for i in range(5):
        m[i, i, i] = 1
    assert CC.label(m, 6)[1] == 5 and CC.label(m, 18)[1] == 5 and CC.label(m, 26)[1] == 1
    m2 = np.zeros((5, 5, 5), np.uint8)
    for i in range(5):
        m2[0, i, i] = 1                                    # a face diagonal: 18 and 26
    assert CC.label(m2, 6)[1] == 5 and CC.label(m2, 18)[1] == 1 and CC.label(m2, 26)[1] == 1


def test_ties_go_to_the_lower_label():
    m = np.zeros((3, 8, 8), np.uint8)
    m[0, 0, 4:7] = 1                                       # label 1, 3 voxels
    m[2, 5, 0:3] = 1                                       # label 2, 3 voxels
    m[1, 7, 7] = 1                                         # label 3 (first voxel after label 1's, before label 2's)
    lab, n = CC.label(m, 6)
    assert n == 3 and lab[0, 0, 4] == 1 and lab[1, 7, 7] == 2 and lab[2, 5, 0] == 3
    out = CC.largest(m, 6)
    assert out.sum() == 3 and out[0, 0, 4:7].all()
    assert np.array_equal(CC.remove_small(m, 2, 6), m * (lab != 2))
    assert np.array_equal(CC.remove_small(m, 0, 6), m)


def test_filters_keep_input_values_and_dtype():
    m = np.zeros((2, 4, 4), np.float32)
    m[0, 0, 0:3] = [1.0, 2.0, 2.0]
    m[1, 3, 3] = 2.0
    out = CC.largest(m, 26)
    assert out.dtype == np.float32 and np.array_equal(out[0, 0, 0:3], [1.0, 2.0, 2.0]) and out[1, 3, 3] == 0
    b = m != 0
    assert CC.largest(b, 26).dtype == np.bool_


def test_batches_are_labelled_on_their_own():
    m = np.zeros((2, 3, 4, 4), np.uint8)
    m[0, 2] = 1                                            # last plane of volume 0
    m[1, 0] = 1                                            # first plane of volume 1
    m[1, 2, 0, 0] = 1
    lab, counts = CC.label(m, 26)
    assert counts.tolist() == [1, 2] and lab[0].max() == 1 and lab[1].max() == 2
    for b in range(2):
        assert np.array_equal(lab[b], CC.label(m[b], 26)[0])
    out = CC.largest(m, 26)
    assert np.array_equal(out[0], m[0]) and out[1, 2, 0, 0] == 0 and out[1, 0].all()


def test_argument_errors_without_a_device():
    m = torch.zeros(4, 4, 4, dtype=torch.uint8)
    for fn in (P.label_components, P.largest_component, lambda t: P.remove_small_components(t, 3)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(m)
        with pytest.raises(ValueError):
            fn(torch.zeros(4, 4, dtype=torch.uint8))                       # rank
        with pytest.raises(ValueError):
            fn(torch.zeros(1, 1, 4, 4, 4, dtype=torch.uint8))
        with pytest.raises(TypeError):
            fn(torch.zeros(4, 4, 4, dtype=torch.int16))
        with pytest.raises(ValueError):
            fn(torch.zeros(1, dtype=torch.uint8).expand(2 ** 11, 2 ** 10, 2 ** 10))   # 2^31 voxels
    for conn in (0, 4, 8, 27, "6"):
        with pytest.raises(ValueError):
            P.label_components(m, conn)
        with pytest.raises(ValueError):
            P.largest_component(m, conn)
    with pytest.raises(ValueError):
        P.remove_small_components(m, -1)
    with pytest.raises(ValueError):
        P.remove_small_components(m, 2.5)
