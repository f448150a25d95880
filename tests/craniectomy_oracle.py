"""TEST INFRASTRUCTURE ONLY -- the CPU statement of the virtual craniectomy drawn on the device (DESIGN.md section 7f).

The distribution is the reference's ``random_blank_patch(image, p, True, p_type="random", valid_shapes)``
(transforms.py:241-300) per sample; the stream is a Philox4x32-10 on the device instead of the host RNGs, so this file
freezes which Philox word feeds which draw (include/ctunet_b200.h, ctu_craniectomy_draw):

  counter = (pass, sample, call), key = the 64-bit seed; r[call][0..3] the four output words
  call 0: gate u53(r0, r1) (applied iff u <= p and the skull has bone); centre rank k = (r2 | r3 << 32) * n >> 64
  call 1: radius = min_r + ((r0 | r1 << 32) * (max_r - min_r) >> 64); shape rank (r2 | r3 << 32) * n_shapes >> 64
  call 2: c_diam = ((0.25 + 0.75 u53(r0, r1)) * radius) / 4 for the flap (0 otherwise)

  draw(key, pass_, full, p, shapes)   params [B, 7] = (applied, shape, radius, c_diam, z, y, x), float64, bit for bit
  inside(row, vol_shape)              the hole of one params row with the kernels' arithmetic (common.cuh: ball_inside,
                                      flap_hole / flap_inside): integer-exact sphere and box, float64 flap
  cut(full, params)                   (broken, full, flap) uint8 = (full AND NOT inside, full, full AND inside)
  encode(full, params, matrices)      the cut in skull space, then affine_oracle.sample (the fused encoder)
"""
import numpy as np

import affine_oracle as A

SHAPE_CODES = {"sphere": 0, "box": 1, "flap": 2}
SHAPE_NAMES = ("sphere", "box", "flap")


def radius_bounds(vol_shape):
    """utilities.radius_bounds as the integers the kernel takes (transforms.py:266-267)."""
    min_r = int(np.min(vol_shape)) // 5 - 1
    max_r = int(np.max([min_r, np.max(vol_shape) // 3.5]))
    return min_r, max_r


def u53(a, b):
    return ((int(a) >> 5) * 67108864.0 + (int(b) >> 6)) / 9007199254740992.0


def words(key, pass_, batch):
    """uint32 [B, 3, 4]: the Philox words of every (sample, call) of one pass."""
    i = np.arange(batch, dtype=np.uint64)
    out = []
    for call in range(3):
        ctr = np.stack([np.full(batch, pass_ & 0xFFFFFFFF, np.uint64), np.full(batch, pass_ >> 32, np.uint64), i,
                        np.full(batch, call, np.uint64)], axis=-1)
        out.append(A.philox4x32_10(ctr, key))
    return np.stack(out, axis=1)


def pick(word_lo, word_hi, n):
    """floor(r * n / 2^64) for the 64-bit word r = lo | hi << 32."""
    return ((int(word_lo) | (int(word_hi) << 32)) * int(n)) >> 64


def kth_voxel(vol, k):
    """The k-th non-zero voxel of ``vol`` in C order, from the flat index."""
    return tuple(int(c) for c in np.unravel_index(np.flatnonzero(vol)[k], vol.shape))


def shape_mask(shapes):
    return sum({1 << SHAPE_CODES[s] for s in shapes})


def draw(key, pass_, full, p, shapes=SHAPE_NAMES):
    """full: uint8 / bool [B, D, H, W] (non-zero is bone) -> params float64 [B, 7]."""
    full = np.asarray(full)
    b_, vol = full.shape[0], full.shape[1:]
    min_r, max_r = radius_bounds(vol)
    enabled = [c for c in range(3) if (shape_mask(shapes) >> c) & 1]
    r = words(key, pass_, b_)
    out = np.zeros((b_, 7), dtype=np.float64)
    for b in range(b_):
        w0, w1, w2 = r[b]
        n = int(np.count_nonzero(full[b]))
        applied = u53(w0[0], w0[1]) <= p and n > 0
        radius = min_r + pick(w1[0], w1[1], max_r - min_r)
        shape = enabled[pick(w1[2], w1[3], len(enabled))]
        c_diam = ((0.25 + 0.75 * u53(w2[0], w2[1])) * float(radius)) / 4.0 if shape == 2 else 0.0
        centre = kth_voxel(full[b], pick(w0[2], w0[3], n)) if applied else (-1, -1, -1)
        out[b] = (float(applied), shape, radius, c_diam) + centre
    return out


def inside(row, vol_shape):
    """bool [D, H, W]: the voxels inside the hole of one params row (whether or not it is applied)."""
    d, h, w = vol_shape
    shape, size, c_diam = int(row[1]), float(row[2]), float(row[3])
    c = [int(v) for v in row[4:7]]
    z, y, x = np.ogrid[:d, :h, :w]
    if shape in (0, 1):
        r = int(size)
        dz, dy, dx = (z - c[0]).astype(np.int64), (y - c[1]).astype(np.int64), (x - c[2]).astype(np.int64)
        if shape == 0:
            return (dz * dz + dy * dy + dx * dx <= r * r) & (r >= 0)
        return (np.abs(dz) <= r) & (np.abs(dy) <= r) & (np.abs(dx) <= r)
    z0 = np.rint((d - 1) * (c[0] / d))
    ey = np.rint((h - 1) * ((c[1] - size / 2) / h))
    ex1, ex2 = np.rint((w - 1) * ((c[2] - size / 2) / w)), np.rint((w - 1) * ((c[2] + size / 2) / w))
    qy, qx = np.rint((h - 1) * (c[1] / h)), np.rint((w - 1) * (c[2] / w))
    half, r2 = size / 2, c_diam * c_diam
    zf, yf, xf = z.astype(np.float64), y.astype(np.float64), x.astype(np.float64)
    dy2 = (yf - ey) ** 2
    cyl = ((dy2 + (xf - ex1) ** 2) <= r2) | ((dy2 + (xf - ex2) ** 2) <= r2)
    cube = (np.abs(yf - qy) <= half) & (np.abs(xf - qx) <= half)
    return (np.abs(zf - z0) <= half) & (cyl | cube)


def cut(full, params):
    """(broken, full, flap) uint8 [B, D, H, W] of full-skull masks [B, D, H, W] and params [B, 7]."""
    f = np.asarray(full) != 0
    ins = np.stack([inside(p, f.shape[1:]) & bool(p[0]) for p in np.asarray(params)])
    return (f & ~ins).astype(np.uint8), f.astype(np.uint8), (f & ins).astype(np.uint8)


def encode(full, params, matrices=None):
    """What the fused encoder writes as masks: the cut in skull space, then the affine gather of all three."""
    masks = list(cut(full, params))
    return masks if matrices is None else A.sample(masks, matrices)
