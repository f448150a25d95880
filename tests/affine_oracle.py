"""TEST INFRASTRUCTURE ONLY -- the CPU statement of the random affine augmentation (DESIGN.md section 7e).

There is no reference counterpart (the reference has no spatial augmentation): this file freezes the semantics, and parity
with MONAI or scipy is not a goal.

  draw(key, pass_, batch, ranges, flip_axes)  the float32 parameters [B, 10] of ctu_affine_draw, bit for bit: a numpy
                                              Philox4x32-10, 24-bit uniforms, float32 arithmetic in the kernel's order
  matrix_from_params(params, shape)           the float32 [B, 3, 4] maps, built in float64 and rounded once
  sample(masks, matrices)                     nearest-neighbour gather in float32 in the kernel's order (numpy does one
                                              IEEE rounding per operation, never an FMA)
"""
import math

import numpy as np

F = np.float32
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def philox4x32_10(ctr, key):
    """ctr: uint32 [..., 4]; key: 64-bit int -> uint32 [..., 4] (common.cuh: philox4x32_10)."""
    c = [np.asarray(ctr[..., i], dtype=np.uint64) for i in range(4)]
    k0, k1 = key & 0xFFFFFFFF, (key >> 32) & 0xFFFFFFFF
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return np.stack([x.astype(np.uint32) for x in c], axis=-1)


def u24(r):
    return (r >> np.uint32(8)).astype(F) * F(1.0 / 16777216.0)


def ranges_f32(rotate_deg, scale, translate):
    """The float32 ranges the kernel reads (RandomAffine._ranges): radians rounded once."""
    return [F(math.radians(r)) for r in rotate_deg] + [F(scale[0]), F(scale[1])] + [F(t) for t in translate]


def draw(key, pass_, batch, ranges, flip_axes):
    i = np.arange(batch, dtype=np.uint64)
    u = []
    for call in range(3):
        ctr = np.stack([np.full(batch, pass_ & 0xFFFFFFFF, np.uint64), np.full(batch, pass_ >> 32, np.uint64), i,
                        np.full(batch, call, np.uint64)], axis=-1)
        r = philox4x32_10(ctr, key)
        u += [u24(r[:, j]) for j in range(4)]
    rng = [F(x) for x in ranges]
    p = np.zeros((batch, 10), dtype=F)
    for k in range(3):
        p[:, k] = rng[k] * (F(2) * u[k] - F(1))
        p[:, 4 + k] = rng[5 + k] * (F(2) * u[4 + k] - F(1))
        p[:, 7 + k] = np.where(((flip_axes >> k) & 1) & (u[7 + k] < F(0.5)), F(-1), F(1))
    p[:, 3] = rng[3] + (rng[4] - rng[3]) * u[3]
    return p


def rotation(a_d, a_h, a_w):
    """R = R_d(a_d) R_h(a_h) R_w(a_w) on (z, y, x) vectors; R_a rotates about axis a."""
    cd, sd, ch, sh, cw, sw = math.cos(a_d), math.sin(a_d), math.cos(a_h), math.sin(a_h), math.cos(a_w), math.sin(a_w)
    rd = np.array([[1, 0, 0], [0, cd, -sd], [0, sd, cd]])
    rh = np.array([[ch, 0, sh], [0, 1, 0], [-sh, 0, ch]])
    rw = np.array([[cw, -sw, 0], [sw, cw, 0], [0, 0, 1]])
    return rd @ rh @ rw


def matrix_from_params(params, shape):
    """q = c + t + (1/s) R F (p - c), c = (S - 1) / 2, as float32 [B, 3, 4] = [A | c + t - A c], A = R F / s."""
    params = np.asarray(params, dtype=np.float64).reshape(-1, 10)
    c = (np.asarray(shape, dtype=np.float64) - 1) / 2
    out = np.zeros((params.shape[0], 3, 4), dtype=np.float64)
    for b, p in enumerate(params):
        a = rotation(p[0], p[1], p[2]) * p[7:10][None, :] / p[3]
        out[b, :, :3] = a
        out[b, :, 3] = c + p[4:7] - a @ c
    return out.astype(F)


def sample(masks, matrices):
    """masks: list of uint8 [B, D, H, W] (numpy); matrices float32 [B, 3, 4] -> the transformed masks (uint8)."""
    b_, d, h, w = masks[0].shape
    z, y, x = [v.astype(F) for v in np.meshgrid(np.arange(d), np.arange(h), np.arange(w), indexing="ij")]
    lim = (F(d) - F(0.5), F(h) - F(0.5), F(w) - F(0.5))
    outs = [np.zeros_like(m) for m in masks]
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(b_):
            m = np.asarray(matrices[b], dtype=F)
            inside = np.ones((d, h, w), dtype=bool)
            idx = []
            for k in range(3):
                q = ((m[k, 0] * z + m[k, 1] * y) + m[k, 2] * x) + m[k, 3]
                inside &= (q > F(-0.5)) & (q < lim[k])
                idx.append(np.floor(q + F(0.5)))
            iz, iy, ix = [np.where(inside, i, 0).astype(np.int64) for i in idx]
            for src, dst in zip(masks, outs):
                dst[b] = np.where(inside, src[b][iz, iy, ix], 0)
    return outs


def identity(batch):
    return np.tile(np.eye(3, 4, dtype=F), (batch, 1, 1))
