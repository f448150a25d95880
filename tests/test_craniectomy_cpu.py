"""CPU: the device craniectomy's oracle (tests/craniectomy_oracle.py) checked against its documented Philox word order,
np.argwhere, the reference's blank_patch (oracle/unet_oracle.py) and the affine oracle; the key derivation; and the argument
errors of the Python surface and the C ABI (no GPU needed: every error comes before a launch)."""
import numpy as np
import pytest
import torch

import affine_oracle as A
import craniectomy_oracle as K
from oracle import unet_oracle as O


def _skulls(b, shape, seed, density=0.3):
    g = np.random.default_rng(seed)
    return (g.random((b,) + shape) < density).astype(np.uint8)


def test_draws_follow_the_documented_philox_words():
    key, pass_ = 0x0123_4567_89AB_CDEF, (5 << 32) | 7
    full = _skulls(6, (12, 14, 16), 0)
    full[3] = 0                                                           # an empty skull
    shapes = ("sphere", "flap")
    params = K.draw(key, pass_, full, 0.7, shapes)
    min_r, max_r = K.radius_bounds((12, 14, 16))
    for b in range(6):
        r = [A.philox4x32_10(np.array([[pass_ & 0xFFFFFFFF, pass_ >> 32, b, call]], dtype=np.uint32), key)[0]
             for call in range(3)]
        u = ((int(r[0][0]) >> 5) * 2.0 ** 26 + (int(r[0][1]) >> 6)) / 2.0 ** 53
        n = int(full[b].sum())
        applied = u <= 0.7 and n > 0
        assert params[b, 0] == float(applied)
        radius = min_r + ((int(r[1][0]) + (int(r[1][1]) << 32)) * (max_r - min_r) >> 64)
        assert params[b, 2] == radius
        shape = (0, 2)[(int(r[1][2]) + (int(r[1][3]) << 32)) * 2 >> 64]
        assert params[b, 1] == shape
        uc = ((int(r[2][0]) >> 5) * 2.0 ** 26 + (int(r[2][1]) >> 6)) / 2.0 ** 53
        assert params[b, 3] == (np.float64(np.float64(0.25) + np.float64(0.75) * uc) * radius / 4 if shape == 2 else 0.0)
        if applied:
            k = (int(r[0][2]) + (int(r[0][3]) << 32)) * n >> 64
            assert tuple(params[b, 4:]) == tuple(np.argwhere(full[b] > 0)[k])
        else:
            assert tuple(params[b, 4:]) == (-1, -1, -1)
    assert params[3, 0] == 0
    assert not np.array_equal(params, K.draw(key, pass_ + 1, full, 0.7, shapes))


@pytest.mark.parametrize("shape", [(5, 6, 7), (3, 1, 9)])
def test_kth_voxel_is_argwhere(shape):
    vol = _skulls(1, shape, 1, 0.4)[0]
    ref = np.argwhere(vol > 0)
    assert len(ref) > 0
    for k in range(len(ref)):
        assert K.kth_voxel(vol, k) == tuple(ref[k])


def _rows(vol_shape, seed, n=24):
    g = np.random.default_rng(seed)
    rows = []
    for i in range(n):
        shape = i % 3
        radius = int(g.integers(-1, max(vol_shape) // 2))
        c_diam = (0.25 + 0.75 * g.random()) * radius / 4 if shape == 2 else 0.0
        centre = [int(g.integers(0, s)) for s in vol_shape]
        rows.append([1.0, shape, radius, c_diam] + centre)
    return np.array(rows, dtype=np.float64)


@pytest.mark.parametrize("vol_shape", [(16, 20, 24), (9, 13, 7)])
def test_masks_equal_blank_patch(vol_shape):
    """Sphere and box (integer-exact) and the flap (float64) against unet_oracle.blank_patch for given draws, including
    radius -1 (nothing inside) and 0 (the centre only)."""
    rows = _rows(vol_shape, 2)
    rows[0, 1:3] = (0, -1)
    rows[1, 1:3] = (1, 0)
    full = _skulls(len(rows), vol_shape, 3, 0.5)
    broken, full01, flap = K.cut(full, rows)
    for b, row in enumerate(rows):
        m, e = O.blank_patch(full[b], [int(c) for c in row[4:]], row[2], K.SHAPE_NAMES[int(row[1])],
                             row[3] if row[1] == 2 else None)
        assert np.array_equal(broken[b], m) and np.array_equal(flap[b], e), row
    assert flap[0].sum() == 0 and flap[1].sum() <= 1
    assert np.array_equal(full01, full)


def test_not_applied_leaves_the_skull_whole():
    full = _skulls(2, (8, 8, 8), 4, 0.5)
    rows = _rows((8, 8, 8), 5, 2)
    rows[:, 0] = 0
    broken, f, flap = K.cut(full, rows)
    assert np.array_equal(broken, full) and flap.sum() == 0


def test_composed_with_affine_equals_hole_then_affine():
    vol = (12, 14, 16)
    full = _skulls(4, vol, 6, 0.4)
    params = K.draw(99, 3, full, 1.0)
    g = np.random.default_rng(7)
    p = np.zeros((4, 10))
    p[:, :3] = np.radians(g.uniform(-30, 30, (4, 3)))
    p[:, 3] = g.uniform(0.8, 1.25, 4)
    p[:, 4:7] = g.uniform(-3, 3, (4, 3))
    p[:, 7:] = np.where(g.random((4, 3)) < 0.5, -1.0, 1.0)
    mats = A.matrix_from_params(p.astype(np.float32), vol)
    cut = [np.stack(t) for t in zip(*[O.blank_patch(full[b], [int(c) for c in params[b, 4:]], params[b, 2],
                                                    K.SHAPE_NAMES[int(params[b, 1])],
                                                    params[b, 3] if params[b, 1] == 2 else None) + (full[b],)
                                      for b in range(4)])]
    ref = A.sample([cut[0], cut[2], cut[1]], mats)
    out = K.encode(full, params, mats)
    assert all(np.array_equal(o, r) for o, r in zip(out, ref))
    assert all(np.array_equal(o, r) for o, r in zip(K.encode(full, params), [cut[0], cut[2], cut[1]]))


def test_mask_invariants():
    vol = (10, 12, 14)
    full = _skulls(8, vol, 8, 0.5)
    full[2] = 0
    params = K.draw(1234, 0, full, 0.6)
    broken, f, flap = K.cut(full, params)
    assert not np.any(broken & flap) and np.array_equal(broken | flap, f)
    assert flap[2].sum() == 0 and params[2, 0] == 0
    applied = params[:, 0] == 1
    assert all(flap[b].sum() > 0 for b in np.flatnonzero(applied) if params[b, 2] >= 0)     # the centre is bone


def test_keys_new_domain_old_keys_unchanged(monkeypatch):
    from ctunet_b200 import engine as E
    from ctunet_b200.utilities import AFFINE_DOMAIN, CRANIECTOMY_DOMAIN
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    torch.manual_seed(1234)
    seed = torch.initial_seed()
    assert E.philox_key("cuda:0") == E._splitmix64(seed ^ E._splitmix64(0))                       # Dropout3d
    assert E.philox_key("cuda:0", AFFINE_DOMAIN) == E._splitmix64(seed ^ E._splitmix64(0 ^ 0xAFF1))  # affine
    assert CRANIECTOMY_DOMAIN not in (0, AFFINE_DOMAIN)
    keys = {E.philox_key("cuda:%d" % dev, dom) for dev in (0, 1) for dom in (0, AFFINE_DOMAIN, CRANIECTOMY_DOMAIN)}
    assert len(keys) == 6


@pytest.mark.parametrize("kw", [dict(p=-0.1), dict(p=1.5), dict(p="1"), dict(shapes=()), dict(shapes="sphere"),
                                dict(shapes=("sphere", "cone"))])
def test_random_craniectomy_argument_errors(kw):
    from ctunet_b200 import RandomCraniectomy
    with pytest.raises(ValueError):
        RandomCraniectomy(**kw)


def test_python_argument_errors_without_a_gpu(monkeypatch):
    from ctunet_b200 import RandomCraniectomy
    from ctunet_b200 import utilities as U
    rc = RandomCraniectomy()
    m = torch.zeros(2, 8, 8, 8, dtype=torch.uint8)
    with pytest.raises(RuntimeError):
        rc.draw(m)                                                  # CPU tensor
    with pytest.raises(TypeError):
        rc.draw(m.float())
    with pytest.raises(ValueError):
        rc.draw(m[0, 0])
    with pytest.raises(ValueError):
        rc.draw(m.view(2, -1), (8, 8, 4))                           # bits of another volume shape
    with pytest.raises(ValueError):
        rc.draw(m.view(2, -1)[:, :64].bool(), (8, 8, 8))            # bit-packed skulls are uint8
    with pytest.raises(ValueError):
        rc.draw(torch.zeros(1, 8, 8, 16385, dtype=torch.uint8))
    with pytest.raises(TypeError):
        rc({"image": m.float()})
    monkeypatch.setattr(U, "radius_bounds", lambda shape: (3, 3))
    with pytest.raises(ValueError, match="empty"):
        rc.draw(m)
    assert rc.last is None


def test_abi_argument_errors_return_negative_without_a_gpu():
    from ctunet_b200 import _lib
    lib = _lib.load()
    fake = 256                                                     # never dereferenced: every call fails its checks first
    ws = lib.ctu_craniectomy_workspace_bytes(2, 8, 8, 8)
    assert ws == 16 and lib.ctu_craniectomy_workspace_bytes(0, 8, 8, 8) == -1
    assert lib.ctu_craniectomy_workspace_bytes(1, 16385, 8, 8) == -1
    assert lib.ctu_craniectomy_workspace_bytes(3, 64, 64, 65) == 784          # 3 x 65 int32 chunk counts, 16-byte rounded
    ok = [0, fake, 2, 8, 8, 8, 1.0, 7, 0, 2, 1, None, fake, fake, ws, None]

    def draw(**kw):
        args = list(ok)
        for i, v in kw.items():
            args[int(i[1:])] = v
        return lib.ctu_craniectomy_draw(*args)
    assert draw(a0=2) < 0                                          # format flag
    assert draw(a1=None) < 0
    assert draw(a2=0) < 0
    assert draw(a5=16385) < 0
    assert draw(a6=1.01) < 0 and draw(a6=-0.5) < 0 and draw(a6=float("nan")) < 0
    assert draw(a7=0) < 0 and draw(a7=8) < 0
    assert draw(a8=2) < 0 and draw(a8=3) < 0                       # empty radius range
    assert draw(a12=None) < 0 and draw(a13=None) < 0
    assert draw(a14=ws - 1) < 0 and draw(a13=fake + 4) < 0         # small / misaligned workspace
    assert draw(a12=fake + 4) < 0                                  # misaligned params
    assert "ctu_craniectomy_draw" in _lib.last_error()
    args = [fake] * 7
    assert lib.ctu_craniectomy_encode_flaprec(2, fake, fake, fake, None, *args[:3], 2, 1, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_encode_flaprec(0, fake, fake, fake, None, *args[:3], 2, 3, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_encode_flaprec(0, fake, fake, None, None, *args[:3], 2, 2, 8, 8, 8, None) < 0   # no atlas
    assert lib.ctu_craniectomy_encode_flaprec(0, fake, None, fake, None, *args[:3], 2, 1, 8, 8, 8, None) < 0   # no params
    assert lib.ctu_craniectomy_encode_flaprec(0, fake, fake, fake, None, fake, None, fake, 2, 1, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_encode_flaprec(0, fake, fake, fake, None, *args[:3], 0, 1, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_masks_u8(fake, fake, fake, fake, None, 2, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_masks_u8(fake, None, fake, fake, fake, 2, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_masks_u8(fake, fake, fake, fake, fake, 2, 0, 8, 8, None) < 0
    assert lib.ctu_craniectomy_masks_u8(fake, fake + 4, fake, fake, fake, 2, 8, 8, 8, None) < 0
    assert lib.ctu_craniectomy_encode_flaprec(0, fake, fake + 4, fake, None, *args[:3], 2, 1, 8, 8, 8, None) < 0
    assert "ctu_craniectomy" in _lib.last_error()
