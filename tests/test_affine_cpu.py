"""CPU: the random affine augmentation's oracle (tests/affine_oracle.py) checked against itself and numpy, the key
derivation, and the argument errors of the Python surface and the C ABI (no GPU needed: every error comes before a launch)."""
import math

import numpy as np
import pytest
import torch

import affine_oracle as A


def _masks(shape, seed):
    g = np.random.default_rng(seed)
    full = (g.random(shape) < 0.4).astype(np.uint8)
    flap = full & (g.random(shape) < 0.3).astype(np.uint8)
    return full - flap, full, flap


def _params(batch, seed, rot=30.0, scale=(0.8, 1.25), shift=6.0):
    g = np.random.default_rng(seed)
    p = np.zeros((batch, 10))
    p[:, :3] = np.radians(g.uniform(-rot, rot, (batch, 3)))
    p[:, 3] = g.uniform(*scale, batch)
    p[:, 4:7] = g.uniform(-shift, shift, (batch, 3))
    p[:, 7:] = np.where(g.random((batch, 3)) < 0.5, -1.0, 1.0)
    return p.astype(np.float32)


def _identity_params(batch):
    p = np.zeros((batch, 10), dtype=np.float32)
    p[:, 3] = 1
    p[:, 7:] = 1
    return p


@pytest.mark.parametrize("shape", [(2, 8, 10, 12), (1, 7, 5, 9)])
def test_identity_is_a_copy(shape):
    m = _masks(shape, 0)
    mats = A.matrix_from_params(_identity_params(shape[0]), shape[1:])
    assert np.array_equal(mats, A.identity(shape[0]))
    for a, b in zip(A.sample(list(m), mats), m):
        assert np.array_equal(a, b)


def test_integer_translation_is_a_zero_filled_shift():
    shape = (1, 9, 10, 11)
    (m,) = _masks(shape, 1)[:1]
    p = _identity_params(1)
    p[0, 4:7] = (2, -3, 1)                 # the source of output p is p + t
    out = A.sample([m], A.matrix_from_params(p, shape[1:]))[0]
    ref = np.zeros_like(m)
    ref[0, :-2, 3:, :-1] = m[0, 2:, :-3, 1:]
    assert np.array_equal(out, ref)


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_flip_is_np_flip(axis):
    shape = (2, 6, 7, 8)
    m = _masks(shape, 2)[1]
    p = _identity_params(2)
    p[:, 7 + axis] = -1
    out = A.sample([m], A.matrix_from_params(p, shape[1:]))[0]
    assert np.array_equal(out, np.flip(m, axis + 1))


@pytest.mark.parametrize("n", [8, 9])
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_quarter_turns_are_rot90(n, axis):
    """A 90 degree turn about one axis of an even or odd cube equals np.rot90 of the plane it rotates."""
    m = _masks((1, n, n, n), 3)[1]
    p = _identity_params(1)
    p[0, axis] = np.float32(math.pi / 2)
    out = A.sample([m], A.matrix_from_params(p, (n, n, n)))[0][0]
    plane = [(1, 2), (0, 2), (0, 1)][axis]
    # about the centre, the source of (y, x) under R_d is (-x, y); of (z, x) under R_h (x, -z); of (z, y) under R_w (-y, z)
    ref = np.rot90(m[0], 1 if axis == 1 else -1, plane)
    assert np.array_equal(out, ref), axis


def test_mask_invariants_survive_random_matrices():
    shape = (6, 12, 14, 16)
    broken, full, flap = _masks(shape, 4)
    mats = A.matrix_from_params(_params(6, 5), shape[1:])
    b2, f2, l2 = A.sample([broken, full, flap], mats)
    assert not np.any(b2 & l2)
    assert np.array_equal(b2 | l2, f2)
    assert 0 < f2.sum() < full.sum() * 2


def test_non_finite_source_reads_zero():
    shape = (3, 5, 6, 7)
    m = np.ones(shape, dtype=np.uint8)
    mats = A.identity(3)
    mats[0, 0, 3] = np.nan
    mats[1, 1, 1] = np.inf
    mats[2, 2, 3] = np.float32(3e38)
    out = A.sample([m], mats)[0]
    assert out[0].sum() == 0 and out[2].sum() == 0
    assert out[1].sum() == 0                        # inf * 0 = NaN at y = 0, inf elsewhere
    assert np.array_equal(A.sample([m], A.identity(3))[0], m)


def test_draw_ranges_and_identity():
    p = A.draw(0x1234_5678_9ABC_DEF0, 7, 4096, A.ranges_f32((15, 10, 5), (0.9, 1.1), (8, 4, 2)), 0b100)
    for k, r in enumerate((15, 10, 5)):
        assert np.abs(p[:, k]).max() <= np.float32(math.radians(r))
    assert p[:, 3].min() >= np.float32(0.9) and p[:, 3].max() <= np.float32(1.1)
    for k, t in enumerate((8, 4, 2)):
        assert np.abs(p[:, 4 + k]).max() <= t
    assert set(np.unique(p[:, 7:9])) == {1.0} and set(np.unique(p[:, 9])) == {-1.0, 1.0}
    q = A.draw(0x1234_5678_9ABC_DEF0, 8, 4096, A.ranges_f32((15, 10, 5), (0.9, 1.1), (8, 4, 2)), 0b100)
    assert not np.array_equal(p, q)
    i = A.draw(99, 0, 16, A.ranges_f32((0, 0, 0), (1, 1), (0, 0, 0)), 0)
    assert np.array_equal(A.matrix_from_params(i, (9, 8, 7)), A.identity(16))


def test_keys_are_distinct_and_the_dropout_key_is_unchanged(monkeypatch):
    from ctunet_b200 import engine as E
    from ctunet_b200.utilities import AFFINE_DOMAIN
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    torch.manual_seed(1234)
    seed = torch.initial_seed()
    old = E._splitmix64(seed ^ E._splitmix64((0 << 32) | 0))          # DropoutRNG's key before the domain existed
    assert E.philox_key("cuda:0") == old
    keys = {E.philox_key("cuda:%d" % dev, dom) for dev in (0, 1) for dom in (0, AFFINE_DOMAIN)}
    assert len(keys) == 4
    monkeypatch.setattr(torch.distributed, "is_initialized", lambda: True)
    monkeypatch.setattr(torch.distributed, "get_rank", lambda: 3)
    assert E.philox_key("cuda:0", AFFINE_DOMAIN) not in keys
    assert E.philox_key("cuda:0") == E._splitmix64(seed ^ E._splitmix64(3))


@pytest.mark.parametrize("kw,exc", [
    (dict(rotate=-1), ValueError), (dict(rotate=181), ValueError), (dict(rotate=(1, 2)), ValueError),
    (dict(rotate=float("nan")), ValueError), (dict(scale=(1.1, 0.9)), ValueError), (dict(scale=(0, 1)), ValueError),
    (dict(scale=1.0), ValueError), (dict(translate=-2), ValueError), (dict(flip=(True,)), ValueError),
    (dict(flip=(1, 0, 0)), ValueError),
])
def test_random_affine_argument_errors(kw, exc):
    from ctunet_b200 import RandomAffine
    with pytest.raises(exc):
        RandomAffine(**kw)


def test_python_argument_errors_without_a_gpu():
    from ctunet_b200 import RandomAffine, affine_masks
    m = torch.zeros(2, 4, 4, 4, dtype=torch.uint8)
    mats = torch.zeros(2, 3, 4)
    with pytest.raises(RuntimeError):
        affine_masks([m], mats)                                     # CPU tensors
    with pytest.raises(TypeError):
        affine_masks([m.float()], mats)
    with pytest.raises(ValueError):
        affine_masks([m, m[:1]], mats)
    with pytest.raises(ValueError):
        affine_masks([m] * 4, mats)
    with pytest.raises(ValueError):
        affine_masks([m[0]], mats)
    with pytest.raises(RuntimeError):
        RandomAffine().draw(2, (4, 4, 4), "cpu")
    with pytest.raises(ValueError):
        RandomAffine()({"image": m.float(), "target": m})


def test_abi_argument_errors_return_negative_without_a_gpu():
    from ctunet_b200 import _lib
    lib = _lib.load()
    fake = 256                                                     # never dereferenced: every call fails its checks first
    rng = (_lib.c_float * 8)(0.2, 0.2, 0.2, 0.9, 1.1, 8, 8, 8)
    bad_rng = (_lib.c_float * 8)(0.2, 0.2, 0.2, 1.1, 0.9, 8, 8, 8)
    assert lib.ctu_affine_draw(0, 8, 8, 8, rng, 4, 1, None, fake, fake, None) < 0
    assert lib.ctu_affine_draw(2, 8, 8, 8, bad_rng, 4, 1, None, fake, fake, None) < 0
    assert lib.ctu_affine_draw(2, 8, 8, 8, rng, 8, 1, None, fake, fake, None) < 0
    assert lib.ctu_affine_draw(2, 8, 8, 8, None, 4, 1, None, fake, fake, None) < 0
    assert lib.ctu_affine_draw(2, 1 << 22, 8, 8, rng, 4, 1, None, fake, fake, None) < 0
    args = [fake] * 8
    assert lib.ctu_affine_encode_flaprec(2, *args, 2, 1, 8, 8, 8, None) < 0      # format flag
    assert lib.ctu_affine_encode_flaprec(0, *args, 2, 3, 8, 8, 8, None) < 0      # channels
    assert lib.ctu_affine_encode_flaprec(0, fake, fake, fake, None, *args[:5], 2, 2, 8, 8, 8, None) < 0   # no atlas
    assert lib.ctu_affine_encode_flaprec(0, *args[:5], None, fake, fake, 2, 1, 8, 8, 8, None) < 0        # null image
    assert lib.ctu_affine_encode_flaprec(0, *args, 0, 1, 8, 8, 8, None) < 0
    assert lib.ctu_affine_encode_flaprec(0, *args, 2, 1, 0, 8, 8, None) < 0
    src = _lib.ptr_array([fake] * 3)
    assert lib.ctu_affine_masks_u8(0, src, src, fake, 2, 8, 8, 8, None) < 0
    assert lib.ctu_affine_masks_u8(4, src, src, fake, 2, 8, 8, 8, None) < 0
    assert lib.ctu_affine_masks_u8(2, _lib.ptr_array([fake, None]), src, fake, 2, 8, 8, 8, None) < 0
    assert lib.ctu_affine_masks_u8(1, src, src, None, 2, 8, 8, 8, None) < 0
    assert lib.ctu_affine_masks_u8(1, src, src, fake, 70000, 8, 8, 8, None) < 0
    assert "ctu_affine" in _lib.last_error()
