"""CPU helpers of the bit-exact convolution tests (test_conv_exact_cpu.py, test_gpu_conv_exact.py).

Operands are small integers.  Every bf16 operand is then exact, and so is every product and every fp32 partial sum as long
as the sum of the absolute values of the terms stays below 2^24 (``exact_premise``): the result no longer depends on
summation order, tensor-core accumulation order or atomic order.  A kernel's fp32 output must then equal the float32 CPU
reference bit for bit, and a bf16 output must equal its round-to-nearest-even.
"""
from __future__ import annotations

import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import upfuse_oracle as U  # noqa: E402

EXACT_LIMIT = 2 ** 24
TILE = 16          # the 16 x 16 plane tiles of conv_tc.cu (TC_TH x TC_TW)


# ------------------------------------------------------------------ operand families
def ternary(shape, g: torch.Generator, density: float = 0.5) -> torch.Tensor:
    """Family T: values in {-1, 0, 1}; ``density`` is the probability of a non-zero."""
    nz = torch.rand(shape, generator=g) < density
    sign = torch.randint(0, 2, shape, generator=g).float() * 2 - 1
    return sign * nz.float()


def ternary_bias(c: int, g: torch.Generator) -> torch.Tensor:
    return torch.randint(-2, 3, (c,), generator=g).float()


def small_nonneg(shape, g: torch.Generator) -> torch.Tensor:
    """Family P: values in {0..3}: sums land mostly above 256, where bf16 rounds (ties included)."""
    return torch.randint(0, 4, shape, generator=g).float()


def operand(family: str, shape, g: torch.Generator, density: float = 0.5) -> torch.Tensor:
    if family == "T":
        return ternary(shape, g, density)
    if family == "P":
        return small_nonneg(shape, g)
    raise ValueError(family)


def bias_operand(family: str, c: int, g: torch.Generator) -> torch.Tensor:
    return ternary_bias(c, g) if family == "T" else torch.randint(0, 4, (c,), generator=g).float()


def round_bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 (round to nearest, ties to even) and back to float32."""
    return t.to(torch.bfloat16).to(torch.float32)


# ------------------------------------------------------------------ the integer premise
def _premise(bound: float, what: str) -> float:
    assert bound < EXACT_LIMIT, "%s: the integer premise fails (sum of |terms| up to %.0f >= 2^24)" % (what, bound)
    return bound


def exact_premise(op: str, x=None, w=None, b=None, dy=None, k: int = 3) -> float:
    """Assert that every partial sum of the convolution ``op`` stays an exact integer in fp32, and return the bound.

    forward: max of conv(|x|, |w|) + |b|; dgrad: the same with |dy| and the flipped weights; wgrad: max of sum_v |x||dy|.
    A cheap upper bound (max operand times the largest row sum of the weights, or voxels times the operand maxima) is tried
    first; the bound is computed with absolute values only where the cheap one reaches 2^24."""
    if op in ("fwd", "dgrad"):
        a = x if op == "fwd" else dy
        wa = w.abs() if op == "fwd" else w.abs().transpose(0, 1)
        rows = wa.flatten(1).sum(1).max().item()
        bb = b.abs().max().item() if b is not None else 0.0
        cheap = a.abs().max().item() * rows + bb
        if cheap < EXACT_LIMIT:
            return _premise(cheap, op)
        if op == "fwd":
            full = F.conv3d(x.abs(), w.abs(), b.abs() if b is not None else None, 1, k // 2).max().item()
        else:
            full = F.conv3d(dy.abs(), w.abs().flip(2, 3, 4).transpose(0, 1), None, 1, k // 2).max().item()
        return _premise(full, op)
    if op == "wgrad":
        vox = x.shape[0] * x[0, 0].numel()
        cheap = vox * x.abs().max().item() * dy.abs().max().item()
        if cheap < EXACT_LIMIT:
            return _premise(cheap, op)
        return _premise(conv_wgrad(x.abs(), dy.abs(), k).max().item(), op)
    raise ValueError(op)


# ------------------------------------------------------------------ references (float32 is exact under the premise)
def conv_fwd(srcs, w, b, k: int) -> torch.Tensor:
    x = torch.cat(list(srcs), 1) if isinstance(srcs, (list, tuple)) else srcs
    return F.conv3d(x, w, b, 1, k // 2)


def conv_dgrad(dy, w, k: int, chans=None):
    """Data gradient of conv3d(x, w): conv3d(dy, flipped and transposed w).  ``chans``: split it per source."""
    dx = F.conv3d(dy, w.flip(2, 3, 4).transpose(0, 1), None, 1, k // 2)
    return list(dx.split(list(chans), 1)) if chans is not None else dx


def conv_wgrad(x, dy, k: int) -> torch.Tensor:
    """dw[co][ci][tap] = sum over batch and voxels of dy[co][v] * x[ci][v + tap - k//2] (zero outside): one matrix
    product per tap (autograd's CPU weight gradient of conv3d is several times slower at 4 x 128^3)."""
    p = k // 2
    n, ci, d, h, w = x.shape
    co = dy.shape[1]
    xp = F.pad(x, (p, p, p, p, p, p))
    dyt = dy.transpose(0, 1).reshape(co, -1)
    out = torch.empty(co, ci, k, k, k, dtype=x.dtype)
    for a in range(k):
        for b in range(k):
            for c in range(k):
                xs = xp[:, :, a:a + d, b:b + h, c:c + w].transpose(0, 1).reshape(ci, -1)
                out[:, :, a, b, c] = dyt @ xs.t()
    return out


def bias_grad(dy) -> torch.Tensor:
    return dy.double().sum((0, 2, 3, 4)).float()


def stats_ref(y: torch.Tensor, cout: int = None):
    """(sum, sum of squares) in float64 per natural channel of the stored (rounded) output; a phase-major y (``cout`` set)
    is mapped back to its natural channels first."""
    if cout is not None:
        y = U.depth_to_space(y, cout)
    yd = y.double()
    return yd.sum((0, 2, 3, 4)), (yd * yd).sum((0, 2, 3, 4))


# ------------------------------------------------------------------ fused up-sampling stage
def composed_weights(wt, bt, w3, k: int) -> torch.Tensor:
    """The composed low-resolution 3^3 weights [8*cop][cin+1][3][3][3], computed in float64 and rounded to bf16 (what the
    tensor kernels multiply with)."""
    wn = U.compose(wt.double(), bt.double() if bt is not None else None, w3.double(), k)
    return round_bf16(wn.float())


def composed_bias(b3, cout: int) -> torch.Tensor:
    """Bias of the phase-major output: b3 in every phase, pad rows zero."""
    cop = (cout + 7) // 8 * 8
    out = torch.zeros(8, cop)
    out[:, :cout] = b3
    return out.reshape(-1)


def with_ones(srcs):
    """cat(srcs, ones): the all-ones channel carries the transposed convolution's bias."""
    x0 = srcs[0]
    return torch.cat(list(srcs) + [torch.ones(x0.shape[0], 1, *x0.shape[2:])], 1)


def phase_to_natural(y: torch.Tensor, cout: int) -> torch.Tensor:
    """Phase-major [n][q*cop + co][d][h][w] -> natural [n][cout][2d][2h][2w] (q = qd*4 + qh*2 + qw)."""
    return U.depth_to_space(y, cout)


def natural_to_phase(g: torch.Tensor, cout: int) -> torch.Tensor:
    return U.space_to_depth(g, (cout + 7) // 8 * 8)


def structural_support(cin: int, cout: int) -> torch.Tensor:
    """Entries of the composed 3^3 weight [8*cop][cin+1][3][3][3] that are not structurally zero."""
    ones_t = torch.ones(cin, 1, 2, 2, 2, dtype=torch.float64)
    ones_w = torch.ones(cout, 1, 3, 3, 3, dtype=torch.float64)
    return U.compose(ones_t, torch.ones(1, dtype=torch.float64), ones_w, 3) != 0


# ------------------------------------------------------------------ mismatch reporting
def mismatches(got: torch.Tensor, exp: torch.Tensor, limit: int = 5):
    """(count, [description]) of the elements of two [n][c][z][y][x] tensors that differ; each description names the
    voxel, its 16 x 16 plane tile (ty, tx) and its d-plane."""
    diff = got != exp
    count = int(diff.sum())
    out = []
    if count:
        for idx in diff.nonzero()[:limit].tolist():
            n, c, z, y, x = idx
            out.append("(n=%d, c=%d, z=%d, y=%d, x=%d) tile (%d, %d) plane %d: got %r, expected %r"
                       % (n, c, z, y, x, y // TILE, x // TILE, z, got[tuple(idx)].item(), exp[tuple(idx)].item()))
    return count, out


def assert_exact(got: torch.Tensor, exp: torch.Tensor, what: str):
    assert got.shape == exp.shape, "%s: shape %s vs %s" % (what, tuple(got.shape), tuple(exp.shape))
    if got.dim() != 5:
        got, exp = got.reshape(1, 1, 1, 1, -1), exp.reshape(1, 1, 1, 1, -1)
    count, where = mismatches(got, exp)
    assert count == 0, "%s: %d of %d elements differ; first: %s" % (what, count, got.numel(), "; ".join(where))
