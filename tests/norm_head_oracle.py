"""Float64 references of the BatchNorm+ReLU(+MaxPool) kernels (csrc/bn.cu) and the fused head + Dice/CE kernels
(csrc/head.cu, csrc/loss_math.cuh), and error bounds derived from the kernels' arithmetic.

Every reference is plain torch float64 on the operands the kernel actually read (bf16 or fp32 values, natural NCDHW
layout), on whatever device they live: the GPU tests run it there, the CPU tests run the same code on the CPU.  Where a
kernel consumes an intermediate of an earlier kernel -- the fp32 scale / shift / mean / invstd of the finalisation, the
per-sample loss sums, the stored logit gradients -- the reference of the later kernel takes the kernel's value as its
input, so each bound covers one kernel's arithmetic and a wrong intermediate is caught where it is produced.

Notation of the bounds: u = 2^-24 (fp32 unit roundoff), us = 2^-8 for a bf16 output (0 for fp32), gamma(k) = k u / (1 - k u)
bounds the error of a k-deep fp32 sum relative to the sum of |terms|.  Double-precision steps contribute 2^-50 relative.
"""
from __future__ import annotations

import math

import torch

U32 = 2.0 ** -24
U16 = 2.0 ** -8
UD = 2.0 ** -50

BN_THREADS = 256
STAT_VOX_PER_THREAD = 32       # bn_stats_kernel: voxels per thread and grid-stride pass
VOX_PER_THREAD = 4             # mode-0 BatchNorm kernels
REDUCE_CAP = 148 * 4           # bn_bwd: blocks of the reduce pass
HEAD_THREADS = 256
HEAD_LOSS_CAP = 148 * 16       # head_loss_fwd/bwd_launch: blocks over all samples
HEAD_PGRAD_CAP = 148 * 2       # head_param_grad_launch
HEAD_GRID_CAP = 148 * 8        # head_grid


def gamma(k: int) -> float:
    return k * U32 / (1.0 - k * U32)


def cdiv(a: int, b: int) -> int:
    return -(-a // b)


def storage_u(dtype) -> float:
    """Unit roundoff of the storage type of an activation (the rounding of a bf16 output)."""
    return U16 if dtype == torch.bfloat16 else 0.0


def fp32(t: torch.Tensor) -> torch.Tensor:
    """float64 -> the nearest fp32 value (round to nearest even), as float64."""
    return t.float().double()


# ---------------------------------------------------------------------------------------------- layout helpers
def to_phase(x: torch.Tensor) -> torch.Tensor:
    """Natural [n][c][2d][2h][2w] -> phase-major [n][8*cpad][d][h][w] (block q*cb + b, q = qd*4 + qh*2 + qw)."""
    n, c, D, H, W = x.shape
    cpad = (c + 7) // 8 * 8
    g = x.reshape(n, c, D // 2, 2, H // 2, 2, W // 2, 2).permute(0, 3, 5, 7, 1, 2, 4, 6)
    out = torch.zeros(n, 2, 2, 2, cpad, D // 2, H // 2, W // 2, dtype=x.dtype, device=x.device)
    out[:, :, :, :, :c] = g
    return out.reshape(n, 8 * cpad, D // 2, H // 2, W // 2)


def from_phase(y: torch.Tensor, c: int) -> torch.Tensor:
    n, c8, d, h, w = y.shape
    y = y.reshape(n, 2, 2, 2, c8 // 8, d, h, w)[:, :, :, :, :c]
    return y.permute(0, 4, 5, 1, 6, 2, 7, 3).reshape(n, c, 2 * d, 2 * h, 2 * w)


def windows(x: torch.Tensor) -> torch.Tensor:
    """[n][c][2d][2h][2w] -> [n][c][d][h][w][8], the children of each 2x2x2 window in (d, h, w) scan order."""
    n, c, D, H, W = x.shape
    return x.reshape(n, c, D // 2, 2, H // 2, 2, W // 2, 2).permute(0, 1, 2, 4, 6, 3, 5, 7).reshape(
        n, c, D // 2, H // 2, W // 2, 8)


def unwindows(x: torch.Tensor) -> torch.Tensor:
    n, c, d, h, w, _ = x.shape
    return x.reshape(n, c, d, h, w, 2, 2, 2).permute(0, 1, 2, 5, 3, 6, 4, 7).reshape(n, c, 2 * d, 2 * h, 2 * w)


def _ch(v: torch.Tensor) -> torch.Tensor:
    """Per-channel vector -> broadcastable over [n][c][d][h][w]."""
    return v.reshape(1, -1, 1, 1, 1)


# ---------------------------------------------------------------------------------------------- BatchNorm: statistics
def batch_sums(y: torch.Tensor):
    """(sum, sum of squares) per channel in float64: what the producing convolution's epilogue hands the BatchNorm."""
    yd = y.double()
    return yd.sum((0, 2, 3, 4)), (yd * yd).sum((0, 2, 3, 4))


def stats_sum_error(y: torch.Tensor, phases: int = 1):
    """Error bound of ctu_bn_stats' sums: per thread an fp32 sum of STAT_VOX_PER_THREAD voxels per grid-stride pass
    (the grid covers the plane, so one pass), a 5-level fp32 warp tree, then double across warps and blocks:
    gamma(32 + 5) * sum|y| for the sum, gamma(32 + 6) * sum y^2 for the sum of squares (fmaf)."""
    yd = y.double()
    return gamma(STAT_VOX_PER_THREAD + 5) * yd.abs().sum((0, 2, 3, 4)), gamma(STAT_VOX_PER_THREAD + 6) * (yd * yd).sum((0, 2, 3, 4))


def finalize(s, s2, count, weight, bias, eps):
    """Training-mode finalisation in float64: mean, biased variance, invstd, scale = gamma * invstd,
    shift = beta - mean * scale (bn_finalize_kernel / the folded prologue of the forward kernels)."""
    mean = s / count
    var = (s2 / count - mean * mean).clamp_min(0.0)
    invstd = 1.0 / torch.sqrt(var + eps)
    scale = weight.double() * invstd
    shift = bias.double() - mean * scale
    return dict(mean=mean, var=var, invstd=invstd, scale=scale, shift=shift)


def finalize_bounds(fin, weight, bias, count, eps, es=None, es2=None):
    """Bounds of the fp32 ss = scale | shift | mean | invstd.  es / es2: error bounds of the sums (None: exact sums).
      mean  = (float)(s / count)                  : u |mean| + es / count
      var   = s2 / count - mean^2 (double)        : es2 / count + 2 |mean| es / count + (es / count)^2 + 4 * 2^-50 s2 / count
      invstd= (float)(1 / sqrt(var + eps))        : u invstd + invstd * dvar / (var + eps)  (first order is dvar / 2;
                                                    the factor 1 covers the second order while dvar < (var + eps) / 2)
      scale = gamma * invstd (fp32)               : |gamma| dinvstd + 2u |scale|
      shift = beta - meanf * scale (fp32)         : |mean| dscale + |scale| dmean + 3u (|beta| + |mean scale|)"""
    mean, var, invstd, scale = fin["mean"], fin["var"], fin["invstd"], fin["scale"]
    dm_sum = (es / count) if es is not None else torch.zeros_like(mean)
    dv_sum = (es2 / count) if es2 is not None else torch.zeros_like(mean)
    s2c = var + mean * mean
    dvar = dv_sum + 2 * mean.abs() * dm_sum + dm_sum ** 2 + 4 * UD * s2c
    dmean = U32 * mean.abs() + dm_sum
    dinv = U32 * invstd + invstd * dvar / (var + eps)
    dscale = weight.double().abs() * dinv + 2 * U32 * scale.abs()
    dshift = mean.abs() * dscale + scale.abs() * dmean + 3 * U32 * (bias.double().abs() + (mean * scale).abs())
    return dict(mean=dmean, invstd=dinv, scale=dscale, shift=dshift, var=dvar)


def running(rm0, rv0, fin, count, momentum, updates):
    """Running statistics after ``updates`` identical updates with the kernel's recurrence in float64:
    r <- (1 - m) r + m * stat, m = the fp32 momentum, stat = mean | unbiased variance."""
    m = float(torch.tensor(momentum, dtype=torch.float32))
    unb = fin["var"] * count / (count - 1.0) if count > 1 else fin["var"]
    rm, rv = rm0.double(), rv0.double()
    for _ in range(updates):
        rm = (1 - m) * rm + m * fin["mean"]
        rv = (1 - m) * rv + m * unb
    return rm, rv


def running_bounds(rm0, rv0, fin, dfin, count, momentum, updates):
    """Each fp32 update rounds (1 - m), both products and the sum (4u of max(|r|, |stat|)) and takes (float)stat
    (u |stat| + the statistic's own error, times m); earlier errors shrink by (1 - m) <= 1.  Summed over the updates."""
    m = float(torch.tensor(momentum, dtype=torch.float32))
    unb = fin["var"] * count / (count - 1.0) if count > 1 else fin["var"]
    dunb = dfin["var"] * count / max(count - 1.0, 1.0)
    em = updates * (4 * U32 * torch.maximum(rm0.double().abs(), fin["mean"].abs()) + m * (U32 * fin["mean"].abs() + dfin["mean"]))
    ev = updates * (4 * U32 * torch.maximum(rv0.double().abs(), unb.abs()) + m * (U32 * unb.abs() + dunb))
    return em, ev


# ---------------------------------------------------------------------------------------------- BatchNorm: forward
def preact(y, scale, shift):
    """v = y * scale + shift in float64 with the kernel's fp32 scale / shift: the kernel's fmaf rounds this value once."""
    return y.double() * _ch(scale) + _ch(shift)


def bn_forward(y, scale, shift, keep=None):
    """a = k * relu(y * scale + shift); keep: [n][c] Dropout3d keep factors (None: 1)."""
    a = preact(y, scale, shift).clamp_min(0.0)
    if keep is not None:
        a = a * keep.double()[:, :, None, None, None]
    return a


def pool_forward(a):
    return windows(a).amax(-1)


def act_bound(a_ref, dtype, keep=None):
    """|a - a64| for a = round_T(k * max(fmaf(y, scale, shift), 0)): fmaf (u) and the keep product (u) before the storage
    rounding: us |a64| + (1 + us) * 2u |a64|.  (v <= 0 gives exactly 0; a64 >= 0.)  Also the pooled bound: rounding is
    monotone, so the max of the rounded children is the rounded max."""
    us = storage_u(dtype)
    e = (2 if keep is not None else 1) * U32 * a_ref
    return us * a_ref + (1 + us) * e


# ---------------------------------------------------------------------------------------------- BatchNorm: decisions
def gate_ties(v):
    """Voxels whose ReLU gate fp32 rounding can flip: fmaf rounds the exact v once and keeps its sign, unless v underflows
    below half the smallest fp32 subnormal."""
    return (v != 0) & (v.abs() < 2.0 ** -149)


def window_winners(v):
    """(winner [n][c][d][h][w] in 0..7, tie mask) of relu(v) over each window: the first maximum in (d, h, w) order
    (torch.max_pool3d's routing; the kernel's strict '>' scan).  A window is tied when a child other than the winner is
    below the maximum by at most 2^-23 of it: fp32 rounding of the two (u each) can then make them equal, and the kernel
    keeps the earlier.  Children exactly equal to the maximum stay equal in fp32: both pick the first."""
    r = windows(v.clamp_min(0.0))
    win = r.argmax(-1)                                   # first maximum
    mx = r.amax(-1, keepdim=True)
    close = (mx - r > 0) & (mx - r <= 2.0 ** -23 * mx)
    tie = close.any(-1)
    return win, tie


# ---------------------------------------------------------------------------------------------- BatchNorm: backward
def reduce_depth(mode: int, n: int, c: int, d: int, h: int, w: int) -> int:
    """fp32 depth of the reduce pass's per-thread sums (bn_bwd): grid-stride iterations of the capped grid times the
    voxels per thread and iteration (8 children in modes 1-3, 4 voxels in mode 0), plus the 5-level warp tree."""
    cb = (c + 7) // 8
    spatial = d * h * w
    nblk = cdiv(spatial // 8, BN_THREADS) if mode else cdiv(spatial, BN_THREADS * VOX_PER_THREAD)
    gx = min(nblk, cdiv(REDUCE_CAP, cb * n))
    iters = cdiv(nblk, gx)
    return iters * (8 if mode else VOX_PER_THREAD) + 5


def bn_mode(pool: bool, phase_major: bool, d: int, h: int, w: int) -> int:
    if pool:
        return 1
    if phase_major:
        return 2
    return 3 if not (d % 2 or h % 2 or w % 2) else 0


def bn_backward(y, ss, dA, dP, keep=None, winners=None, flip_gate=None, flip_route=None):
    """Reference backward with the kernel's fp32 scale / shift / mean / invstd (ss as float64 [4][c]):
      dz = k * (dA + [child is the window's winner] dP) * [v > 0]
      sums (sum dz, sum dz * xhat), xhat = (y - mean) * invstd
      dy = scale * (dz - mean(dz) - xhat * mean(dz * xhat)), dbeta = sum dz, dgamma = sum dz * xhat.
    ``flip_gate`` / ``flip_route``: masks of voxels / windows where the other branch of the decision is taken (the
    alternative a kernel may legitimately produce at a tied decision)."""
    scale, shift, mean, invstd = ss
    v = preact(y, scale, shift)
    g = dA.double() if dA is not None else torch.zeros_like(v)
    if dP is not None:
        win, _ = window_winners(v) if winners is None else (winners, None)
        onehot = torch.nn.functional.one_hot(win, 8).double()
        if flip_route is not None:
            # the runner-up (largest child other than the winner) takes the routed gradient instead
            r = windows(v.clamp_min(0.0)).masked_fill(onehot.bool(), -1.0)
            alt = torch.nn.functional.one_hot(r.argmax(-1), 8).double()
            onehot = torch.where(flip_route.unsqueeze(-1), alt, onehot)
        g = g + unwindows(onehot * dP.double().unsqueeze(-1))
    if keep is not None:
        g = g * keep.double()[:, :, None, None, None]
    gate = v > 0
    if flip_gate is not None:
        gate = gate ^ flip_gate
    dz = torch.where(gate, g, torch.zeros_like(g))
    xhat = (y.double() - _ch(mean)) * _ch(invstd)
    count = y.numel() / y.shape[1]
    s1 = dz.sum((0, 2, 3, 4))
    s2 = (dz * xhat).sum((0, 2, 3, 4))
    dy = _ch(scale) * (dz - _ch(s1 / count) - xhat * _ch(s2 / count))
    return dict(dz=dz, xhat=xhat, s1=s1, s2=s2, dy=dy, dbeta=s1, dgamma=s2, count=count)


def dy_error_with_ties(y, ss, dA, dP, keep, dy):
    """(reference, |dy - dy64| per element, tie-marked gates, tie-marked windows): at a tied decision the error is to
    the nearer of the two references (either branch is right), everywhere else to the reference's routing."""
    v = preact(y, ss[0], ss[1])
    gate = gate_ties(v)
    win, tie = window_winners(v) if dP is not None else (None, None)
    ref = bn_backward(y, ss, dA, dP, keep, win)
    err = (dy.double() - ref["dy"]).abs()
    nwin = int(tie.sum()) if dP is not None else 0
    if int(gate.sum()) or nwin:
        alt = bn_backward(y, ss, dA, dP, keep, win, flip_gate=gate, flip_route=tie)
        err = torch.minimum(err, (dy.double() - alt["dy"]).abs())
    return ref, err, gate, tie


def bn_backward_bounds(ref, ss, depth, dtype, tie_dz=None):
    """Bounds of the backward kernels.
      reduce sums: dz carries 2 fp32 roundings ((dA + dP) * k), xhat 2 ((y - mean) * invstd), the fmaf 1, then a
        ``depth``-deep fp32 sum (reduce_depth) and double beyond:  e1 = gamma(depth + 2) sum|dz|,
        e2 = gamma(depth + 5) sum|dz xhat|;  plus sum |dz| (and |dz xhat|) over tied decisions (``tie_dz``), whose
        branch may differ.  dbeta / dgamma add the fp32 cast: u |sum|.
      dy = round_T(scale * ((dz - k1) - xhat * k2)), k1 = (float)(sum dz / count), k2 likewise:
        e = |scale| (dk1 + |xhat| dk2 + 6u (|dz| + |m1| + |xhat| |m2|)) + u |dy64|, dk = e / count + u (|m| + e / count)
        (6u: dz 2, xhat 2, the subtraction, product and subtraction 3 more, less the final product counted in u |dy64|)
        bound = us |dy64| + (1 + us) e."""
    scale = ss[0]
    dz, xhat, count = ref["dz"], ref["xhat"], ref["count"]
    e1 = gamma(depth + 2) * dz.abs().sum((0, 2, 3, 4))
    e2 = gamma(depth + 5) * (dz * xhat).abs().sum((0, 2, 3, 4))
    if tie_dz is not None:
        e1 = e1 + tie_dz.abs().sum((0, 2, 3, 4))
        e2 = e2 + (tie_dz * xhat).abs().sum((0, 2, 3, 4))
    m1, m2 = ref["s1"] / count, ref["s2"] / count
    dk1 = e1 / count + U32 * (m1.abs() + e1 / count)
    dk2 = e2 / count + U32 * (m2.abs() + e2 / count)
    e = _ch(scale.abs()) * (_ch(dk1) + xhat.abs() * _ch(dk2)
                            + 6 * U32 * (dz.abs() + _ch(m1.abs()) + xhat.abs() * _ch(m2.abs()))) + U32 * ref["dy"].abs()
    us = storage_u(dtype)
    return dict(dy=us * ref["dy"].abs() + (1 + us) * e,
                dbeta=e1 + U32 * ref["s1"].abs() + UD * ref["s1"].abs(),
                dgamma=e2 + U32 * ref["s2"].abs() + UD * ref["s2"].abs())


# ---------------------------------------------------------------------------------------------- head + loss
HEAD_SOFTMAX, HEAD_SIGMOID, HEAD_SP, HEAD_SP_SOFTMAX = 1, 2, 4, 8


def head_logits(x, w, b):
    """1x1x1 logits: x [n][cin][...] float64, w [cout][cin], b [cout] -> [n][cout][...]."""
    return torch.einsum("nc...,oc->no...", x.double(), w.double()) + b.double().reshape(1, -1, *([1] * (x.dim() - 2)))


def head_chain(lc, flags):
    """head_forward_chain: optional softmax over the logits, optional sigmoid, then the SP encodings
    skull = [s0, s1 + s2], flap = [1 - s1, s1] (and a softmax over each pair for SP_SOFTMAX).  Returns the list of
    predictions the loss sees: [skull, flap] for the SP heads, [out] otherwise."""
    sm = torch.softmax(lc, 1) if flags & HEAD_SOFTMAX else lc
    sg = torch.sigmoid(sm) if flags & HEAD_SIGMOID else sm
    if flags & (HEAD_SP | HEAD_SP_SOFTMAX):
        sk = torch.stack((sg[:, 0], sg[:, 1] + sg[:, 2]), 1)
        fl = torch.stack((1 - sg[:, 1], sg[:, 1]), 1)
        if flags & HEAD_SP_SOFTMAX:
            sk, fl = torch.softmax(sk, 1), torch.softmax(fl, 1)
        return [sk, fl]
    return [sg]


def pair_sums(pred, tgt, softmax_for_dice):
    """Per-sample [n][4] = (sum q t, sum q q, sum t t, CE sum), q = softmax(pred) if softmax_for_dice else pred, CE with
    ``pred`` as logits against the first arg-max of the one-hot target (loss_voxel_fwd)."""
    q = torch.softmax(pred, 1) if softmax_for_dice else pred
    k = tgt.argmax(1, keepdim=True)
    ce = torch.logsumexp(pred, 1) - pred.gather(1, k).squeeze(1)
    dims = tuple(range(1, pred.dim()))
    return torch.stack(((q * tgt).sum(dims), (q * q).sum(dims), (tgt * tgt).sum(dims), ce.sum(dims[:-1])), 1)


def components(sums, spatial, ce_l, dice_l):
    """head_loss_finalize_kernel's comps from [pairs][n][4] sums: [ce_l * CE per pair] + [dice_l * Dice per pair] +
    [total], in float64."""
    nb = sums.shape[1]
    eps = 1e-7
    ce = sums[:, :, 3].sum(1) / (nb * spatial)
    dice = 1 - 2 * ((sums[:, :, 0] + eps) / (sums[:, :, 1] + sums[:, :, 2] + eps)).sum(1) / nb
    out = ([ce_l * c for c in ce] if ce_l else []) + ([dice_l * d for d in dice] if dice_l else [])
    return torch.stack(out + [sum(out)])


def onehot_targets(targets, u8):
    """uint8 class-1 masks [n][...] -> one-hot float64 [n][2][...]; float one-hot targets pass through."""
    if u8:
        m = targets.double()
        return torch.stack((1 - (m != 0).double(), (m != 0).double()), 1)
    return targets.double()


def surrogate_loss(preds, tgts, coefs, softmax_for_dice, kce):
    """A loss whose gradient with respect to the predictions is the kernels' (loss_voxel_bwd): per pair and sample
    kt sum q t + kq / 2 sum q^2 (Dice linearised at the per-sample sums: kt, kq from dice_coefficients) and
    kce * CE.  At exact sums its gradient is that of oracle.unet_oracle's loss (tests/test_norm_head_cpu.py)."""
    total = 0.0
    for p, t, (kt, kq) in zip(preds, tgts, coefs):
        q = torch.softmax(p, 1) if softmax_for_dice else p
        shp = (-1,) + (1,) * (p.dim() - 1)
        total = total + (kt.reshape(shp) * q * t).sum() + (0.5 * kq.reshape(shp) * q * q).sum()
        if kce:
            k = t.argmax(1, keepdim=True)
            total = total + kce * (torch.logsumexp(p, 1) - p.gather(1, k).squeeze(1)).sum()
    return total


def dice_coefficients(sums, nb, g_dice):
    """kt, kq per pair and sample from [pairs][n][4] sums (double, then fp32 as the kernel rounds them)."""
    eps = 1e-7
    N = sums[:, :, 0] + eps
    D = sums[:, :, 1] + sums[:, :, 2] + eps
    kt = fp32(-2.0 / nb / D) * g_dice
    kq = fp32(4.0 / nb * N / (D * D)) * g_dice
    return [(kt[q], kq[q]) for q in range(sums.shape[0])]


def logit_gradients(lc, flags, tgts, sums, softmax_for_dice, ce_l, dice_l, spatial):
    """dlc [n][cout][...] of the fused backward in float64: autograd of the surrogate loss through the head chain, with
    the Dice coefficients from ``sums`` (the kernel's sums in the GPU tests: what ctu_head_loss_bwd reads)."""
    lc = lc.detach().clone().requires_grad_(True)
    nb = lc.shape[0]
    kce = ce_l / (nb * spatial) if ce_l else 0.0
    preds = head_chain(lc, flags)
    loss = surrogate_loss(preds, tgts, dice_coefficients(sums, nb, dice_l), softmax_for_dice, kce)
    (g,) = torch.autograd.grad(loss, lc)
    return g


def logit_error(x, w, b):
    """|lc - lc64| of the fp32 fmaf chain bias + sum_c x_c w_oc (one fmaf per input lane): gamma(cin) * (|b| + sum|x w|)."""
    cin = x.shape[1]
    lam = torch.einsum("nc...,oc->no...", x.double().abs(), w.double().abs()) + b.double().abs().reshape(1, -1, *([1] * (x.dim() - 2)))
    return gamma(cin) * lam


def chain_error(lc, dlc_abs):
    """Bound of the error of every prediction the loss sees, per voxel: the chains are 1-Lipschitz in the max-norm of the
    logits (sigmoid' <= 1/4, a softmax Jacobian row sums to <= 1/2, the SP sums add two sigmoids, the pair softmax
    halves again), so the logit error passes with factor 1; the approximate intrinsics (__expf: 2 + 1.2|x| ulp,
    __fdividef 2 ulp) and the fp32 roundings of the longest chain (SIGMOID|SP_SOFTMAX: sigmoid, sum, pair softmax) add
    (24 + 4 max|lc|) u."""
    return dlc_abs.amax(1) + (24 + 4 * lc.abs().amax(1)) * U32


def loss_sums_bounds(preds, tgts, softmax_for_dice, eps_pred, depth):
    """Bounds of the four per-sample sums of one pair, [n][4].  Each prediction is off by at most ``eps_pred`` (per
    voxel); q = softmax2(pred) is 1/2-Lipschitz and softmax2_fast adds (8 + 2|d|) u (d = the pair's difference),
    so dq <= eps_pred + (8 + 2|d|) u (or eps_pred without the softmax).  Per voxel: |t| dq per class for sum q t,
    (2|q| + dq) dq for sum q^2, the CE term lse - x_k is 2-Lipschitz plus __logf's 2^-21.4 absolute and 8u of its
    arithmetic.  The fp32 accumulation is ``depth`` deep (head_loss_depth): gamma(depth) sum|terms|."""
    p, t = preds, tgts
    if softmax_for_dice:
        q = torch.softmax(p, 1)
        dq = eps_pred.unsqueeze(1) + (8 + 2 * (p[:, 1] - p[:, 0]).abs().unsqueeze(1)) * U32
    else:
        q = p
        dq = eps_pred.unsqueeze(1).expand_as(p)
    dims = tuple(range(1, p.dim()))
    k = t.argmax(1, keepdim=True)
    ce = torch.logsumexp(p, 1) - p.gather(1, k).squeeze(1)
    lse_err = 2 * eps_pred + 2.0 ** -21.4 + 8 * U32 * (torch.logsumexp(p, 1).abs() + p.abs().amax(1))
    g = gamma(depth)
    return torch.stack((
        (t.abs() * dq).sum(dims) + g * (q * t).abs().sum(dims),
        ((2 * q.abs() + dq) * dq).sum(dims) + g * (q * q).sum(dims),
        g * (t * t).sum(dims),
        lse_err.sum(dims[:-1]) + g * ce.abs().sum(dims[:-1])), 1)


def head_loss_depth(n, spatial, per_voxel_terms):
    """fp32 depth of the fused forward's per-thread sums: the grid is capped at ceil(HEAD_LOSS_CAP / n) blocks per
    sample; every thread takes 2 voxels per iteration (1 when ``spatial`` is odd), ``per_voxel_terms`` fmaf / adds each,
    then the 5-level warp tree (double beyond)."""
    per = spatial // 2 if spatial % 2 == 0 else spatial
    gx = min(cdiv(per, HEAD_THREADS), cdiv(HEAD_LOSS_CAP, n))
    iters = cdiv(per, gx * HEAD_THREADS)
    return iters * (2 if spatial % 2 == 0 else 1) * per_voxel_terms + 5


def components_bounds(sums, dsums, spatial, ce_l, dice_l):
    """comps from the sums (double, then fp32 casts, fp32 products by the weights and an fp32 running total):
    dCE = sum dCE_i / (n spatial), dDice = 2 / n sum (dN / D + N dD / D^2) (first order; D >= sum t^2 >> dD), then
    u |c| for each cast and product, and u |total| per addition."""
    nb = sums.shape[1]
    eps = 1e-7
    N = sums[:, :, 0] + eps
    D = sums[:, :, 1] + sums[:, :, 2] + eps
    dce = dsums[:, :, 3].sum(1) / (nb * spatial)
    ddice = 2.0 / nb * (dsums[:, :, 0] / D + N * (dsums[:, :, 1] + dsums[:, :, 2]) / (D * D)).sum(1)
    ref = components(sums, spatial, ce_l, dice_l)
    errs = ([abs(ce_l) * e for e in dce] if ce_l else []) + ([abs(dice_l) * e for e in ddice] if dice_l else [])
    errs = torch.stack(errs)
    errs = errs + 2 * U32 * ref[:-1].abs()
    total = errs.sum() + len(errs) * U32 * ref[-1].abs() + U32 * ref[:-1].abs().sum()
    return torch.cat((errs, total.reshape(1)))


def dlc_bounds(coefs, kce, eps_pred, lc_err, nb):
    """Bound of the fused backward's logit gradients relative to logit_gradients at the kernel's sums.  Per voxel the
    gradient is a sum of (kt, kq, kce) times products of probability-like factors in [0, 2]; its derivative with respect
    to the logits and to the predictions is at most 4 (|kt| + |kq| + kce) in the max-norm, and the fp32 evaluation of the
    backward chain (about 16 roundings and approximate intrinsics of magnitude <= 2 each) adds 64 u (|kt| + |kq| + kce).
    Returns [pairs-summed scale][n][...] broadcastable over the output channels."""
    k = sum(kt.abs() + kq.abs() for kt, kq in coefs) + kce
    shp = (nb,) + (1,) * (eps_pred.dim() - 1)
    return (k.reshape(shp) * (4 * (lc_err + eps_pred) + 64 * U32)).unsqueeze(1)


def dsrc_ref_and_bound(dlc, w, dtype):
    """dsrc[c] = sum_o dlc[o] w[o][c] from the kernel's fp32 dlc: CO fmaf (gamma(CO) sum|terms|), then the storage
    rounding."""
    dlc = dlc.double()
    ref = torch.einsum("no...,oc->nc...", dlc, w.double())
    e = gamma(w.shape[0]) * torch.einsum("no...,oc->nc...", dlc.abs(), w.double().abs())
    us = storage_u(dtype)
    return ref, us * ref.abs() + (1 + us) * e


def param_grad_depth(n, spatial, cin_blocks):
    """fp32 depth of head_param_grad: per-thread grid-stride sum over the capped grid, 5-level warp tree, the fp32 sum
    of the 8 warp partials, and one fp32 atomic per block into dW / db (any order: as deep as the grid)."""
    total = n * spatial
    grid = min(cdiv(total, HEAD_THREADS), HEAD_GRID_CAP, HEAD_PGRAD_CAP)
    return cdiv(total, grid * HEAD_THREADS) + 5 + 8 + grid


def param_grad_ref_and_bound(dlc, x, depth):
    """dW[o][c] = sum dlc[o] x[c], db[o] = sum dlc[o] from the kernel's fp32 dlc, and gamma(depth) sum|terms|."""
    dlc, x = dlc.double(), x.double()
    dims = [0] + list(range(2, x.dim()))
    dw = torch.einsum("no...,nc...->oc", dlc, x)
    db = dlc.sum(dims)
    g = gamma(depth)
    return dw, db, g * torch.einsum("no...,nc...->oc", dlc.abs(), x.abs()), g * dlc.abs().sum(dims)


# ---------------------------------------------------------------------------------------------- comparison
def ratio(got, ref, bound, floor=1e-30):
    """Worst |got - ref| / bound (a zero bound demands an exact result) and the flat index where it occurs."""
    err = (got.double() - ref.double()).abs()
    r = err / bound.double().clamp_min(floor)
    r = torch.where(bound.double() > 0, r, torch.where(err > 0, torch.full_like(r, math.inf), torch.zeros_like(r)))
    idx = int(r.reshape(-1).argmax())
    return float(r.reshape(-1)[idx]), idx
