"""Float64 references of the tail of the captured training step (csrc/optim.cu) and of what the step must produce, for
checking ``TrainStep`` replay by replay (tests/test_gpu_step_replay.py).

  optimizer_update64   torch.optim's single-tensor Adam / AdamW (amsgrad), RMSprop and SGD in float64, on exactly what
                       ``optim_step_kernel`` read, with a per-element bound for that fp32 kernel
  plateau64            torch's ``ReduceLROnPlateau.step`` on the double[10] record of ``FlatOptimizer.sched``
  bn_update_counts     running-statistics updates per BatchNorm and training step, from the CPU oracle's forward
  slot_table           the (name, offset, numel) slices of the flat gradient buffer, from ``named_parameters()`` alone
  noise_floor          the per-tensor gradient bound of the bf16 product against the float oracles (see its docstring)

Notation of the bounds: u = 2^-24 (fp32 unit roundoff), eta = 2^-149 (the absolute error of one fp32 rounding in the
subnormal range).  One fp32 operation returns x (1 + d) with |d| <= u, or x + d' with |d'| <= eta below 2^-126.  A
constant formed in double and stored as fp32 (1 - beta1, lr / bc1, sqrt(bc2), ...) carries one such rounding.  Products
of two first-order terms are covered by a factor 1.01 on every first-order sum.
"""
from __future__ import annotations

import math
from collections import namedtuple

import torch

U32 = 2.0 ** -24
ETA = 2.0 ** -149
SLACK = 1.01
CHUNK = 1024                   # csrc/optim.cu kChunk: one block of optim_step_kernel per 1024 elements of one parameter

KIND_STATES = {"adam": 3, "adamw": 3, "rmsprop": 2, "sgd": 1}
Update = namedtuple("Update", "p states p_err state_errs")


def _sqrt_err(x, e):
    """|sqrt(x + d) - sqrt(x)| for |d| <= e, x >= 0: d / (sqrt(x + d) + sqrt(x)) <= min(sqrt(e), e / sqrt(x))."""
    r = x.sqrt()
    return torch.minimum(e.sqrt(), e / r.clamp_min(1e-300))


def _decayed_grad(p, g, wd):
    """G = g + wd p (torch: grad.add(param, alpha=wd)) and the kernel's error on it: wd_f32 rounds once and fmaf(p,
    wd_f32, g) once more (an unfused product and sum: one more on wd p), |g1 - G| <= u (2.01 |wd p| + |G|) + 2 eta."""
    if wd == 0:
        return g, torch.zeros_like(g)
    G = g.add(p, alpha=wd)
    return G, SLACK * U32 * (2.01 * (wd * p).abs() + G.abs()) + 2 * ETA


def _second_moment(v, G, e_g, beta):
    """V = v beta + (1 - beta) G^2 (torch: mul_(beta).addcmul_(G, G, value=1 - beta)) and the error of the kernel's
    fp32 ``v * beta_f32 + omb_f32 * g * g``: beta_f32 and omb_f32 one rounding each, v beta_f32 one more (2.01 u v beta),
    omb (g g) two more (3.01 u (1 - beta) G^2) plus the propagated 2 |G| e_g + e_g^2, the sum one more (u V).  Three
    roundings can land in the subnormal range: 3 eta.  (A contracted fmaf only removes roundings.)"""
    V = v.mul(beta).addcmul_(G, G, value=1 - beta)
    e = SLACK * (2.01 * U32 * v.abs() * beta + (1 - beta) * (3.01 * U32 * G * G + 2.01 * G.abs() * e_g + e_g * e_g)
                 + U32 * V) + 3 * ETA
    return V, e


def optimizer_update64(kind: str, p, g, states, lr: float, step: int, hyper: dict) -> Update:
    """One update of ``optim_step_kernel`` restated in float64: ``p`` the parameter before the step, ``g`` the gradient as
    it sits in the flat buffer, ``states`` (state0, state1, state2) before the step (None where the kind keeps none),
    ``lr`` = sched[0] and ``step`` = step_count BEFORE the step (the kernel runs update number step + 1), ``hyper`` =
    ``FlatOptimizer.hyper``.  Returns the float64 parameter and states after the step and, for each, a per-element bound
    on |fp32 kernel - float64 reference|.

    The rules are torch.optim's single-tensor implementations (torch 2.11) in float64, operation for operation:

      Adam / AdamW (amsgrad)   m.lerp_(G, 1 - b1); v.mul_(b2).addcmul_(G, G, value=1 - b2); vmax = max(vmax, v);
                               denom = sqrt(vmax) / sqrt(1 - b2^t) + eps; p -= lr / (1 - b1^t) * m / denom
                               (Adam: G = g + wd p; AdamW: p *= 1 - lr wd first, G = g)
      RMSprop                  sq.mul_(a).addcmul_(G, G, value=1 - a); avg = sqrt(sq) + eps;
                               momentum: buf = buf mom + G / avg, p -= lr buf;  else p -= lr G / avg
      SGD                      momentum: buf = G at t = 1, buf mom + G after;  p -= lr buf (or lr G)

    Bounds, Adam / AdamW, from the kernel's roundings in order (each first-order sum times 1.01):
      m      d = fl(g1 - m) (u |G - m| + e_g), t = fl(d omb1) (omb1_f32 and the product: 2 u more), M = fl(m + t) (u |M|):
             e_m = (1 - b1)(e_g + 3.01 u |G - m|) + u |M| + 2 eta
      v      see ``_second_moment``;  vmax = max(s2, v) is exact and 1-Lipschitz, so e_vmax = e_v
      denom  S = sqrtf(vmax): e_S = sqrt-propagation of e_v + u S + eta; / bc2s_f32 (its rounding and the divide: 2 u);
             + eps_f32 (u eps) and the sum (u D):  e_D = e_S / bc2s + 2 u S / bc2s + u eps + u D + eta
      ratio  r = fl(M / D): e_r = e_m / D + |M| e_D / D^2 + u |M| / D + eta
      update U = fl(ss_f32 r), ss = lr / bc1 in double then fp32 (2 u |U| with the product): e_U = ss e_r + 2 u |U| + eta
      param  P = fl(p1 - U): e_P = e_p1 + e_U + u |P| + eta, where AdamW's p1 = fl(p fl(1 - fl(fl(lr) wd))) carries
             e_p1 = |p| u (3.01 lr wd + 2.01 |1 - lr wd|) + eta and Adam's p1 = p is exact.
    RMSprop: e_sq from ``_second_moment``; A = sqrtf(sq) + eps: e_A = sqrt-propagation + u sqrt(sq) + u eps + u A + eta;
      G / A: e_q = e_g / A + |G| e_A / A^2 + u |G / A| + eta; with momentum B = fl(fl(buf mom_f32) + q):
      e_B = 2.01 u |buf mom| + e_q + u |B| + eta; P = fl(p - fl(lr_f32 B)): e_P = lr e_B + 2 u lr |B| + u |P| + eta.
    SGD: B = G (t = 1) or fl(fl(buf mom_f32) + G): e_B = e_g or 2.01 u |buf mom| + e_g + u |B| + eta; P as RMSprop."""
    p, g = p.double(), g.double()
    s = [t.double() if t is not None else None for t in states]
    wd, mom = float(hyper["weight_decay"]), float(hyper["momentum"])
    eps = float(hyper["eps"])
    t = int(step) + 1
    out_s, err_s = [None, None, None], [None, None, None]
    if kind in ("adam", "adamw"):
        b1, b2 = float(hyper["beta1"]), float(hyper["beta2"])
        p1, e_p1 = p, torch.zeros_like(p)
        if kind == "adamw" and wd != 0:
            p1 = p.mul(1 - lr * wd)
            e_p1 = SLACK * p.abs() * U32 * (3.01 * lr * wd + 2.01 * abs(1 - lr * wd)) + ETA
            G, e_g = g, torch.zeros_like(g)
        else:
            G, e_g = _decayed_grad(p, g, wd)
        M = s[0].lerp(G, 1 - b1)
        e_m = SLACK * ((1 - b1) * (e_g + 3.01 * U32 * (G - s[0]).abs()) + U32 * M.abs()) + 2 * ETA
        V, e_v = _second_moment(s[1], G, e_g, b2)
        out_s[0], out_s[1], err_s[0], err_s[1] = M, V, e_m, e_v
        vm = V
        if hyper["amsgrad"]:
            vm = torch.maximum(s[2], V)
            out_s[2], err_s[2] = vm, e_v
        bc1 = 1 - b1 ** t
        bc2s = math.sqrt(1 - b2 ** t)
        ss = lr / bc1
        S = vm.sqrt()
        D = S / bc2s + eps
        e_S = SLACK * (_sqrt_err(vm, e_v) + U32 * S) + ETA
        e_D = SLACK * (e_S / bc2s + 2 * U32 * S / bc2s + U32 * eps + U32 * D) + ETA
        e_r = SLACK * (e_m / D + M.abs() * e_D / (D * D) + U32 * M.abs() / D) + ETA
        U = M / D * ss
        e_U = SLACK * (ss * e_r + 2 * U32 * U.abs()) + ETA
        P = p1.addcdiv(M, D, value=-ss)
        e_P = SLACK * (e_p1 + e_U + U32 * P.abs()) + ETA
        return Update(P, tuple(out_s), e_P, tuple(err_s))
    G, e_g = _decayed_grad(p, g, wd)
    if kind == "rmsprop":
        a = float(hyper["alpha"])
        SQ, e_sq = _second_moment(s[0], G, e_g, a)
        out_s[0], err_s[0] = SQ, e_sq
        R = SQ.sqrt()
        A = R + eps
        e_A = SLACK * (_sqrt_err(SQ, e_sq) + U32 * R + U32 * eps + U32 * A) + ETA
        Q = G / A
        e_q = SLACK * (e_g / A + G.abs() * e_A / (A * A) + U32 * Q.abs()) + ETA
        if mom > 0:
            B = s[1].mul(mom).addcdiv(G, A)
            e_B = SLACK * (2.01 * U32 * (s[1] * mom).abs() + e_q + U32 * B.abs()) + ETA
            out_s[1], err_s[1] = B, e_B
        else:
            P = p.addcdiv(G, A, value=-lr)
            e_P = SLACK * (lr * e_q + 2 * U32 * lr * Q.abs() + U32 * P.abs()) + ETA
            return Update(P, tuple(out_s), e_P, tuple(err_s))
    elif kind == "sgd":
        if mom != 0:
            if t == 1:
                B, e_B = G.clone(), e_g
            else:
                B = s[0].mul(mom).add(G)
                e_B = SLACK * (2.01 * U32 * (s[0] * mom).abs() + e_g + U32 * B.abs()) + ETA
            out_s[0], err_s[0] = B, e_B
        else:
            B, e_B = G, e_g
    else:
        raise ValueError("optimizer kind %r" % kind)
    P = p.add(B, alpha=-lr)
    e_P = SLACK * (lr * e_B + 2 * U32 * lr * B.abs() + U32 * P.abs()) + ETA
    return Update(P, tuple(out_s), e_P, tuple(err_s))


# ---------------------------------------------------------------------------------------------- scheduler
def plateau64(sched, loss) -> torch.Tensor:
    """torch's ``ReduceLROnPlateau.step(loss)`` (mode 'min', threshold_mode 'rel') on the float64 record
    [lr, best, num_bad_epochs, cooldown_counter, factor, patience, threshold, min_lr, cooldown, eps] of
    ``FlatOptimizer.sched``.  ``loss`` is the fp32 total the step computed; ``optim_post_kernel`` widens it to double and
    applies the same double operations, so the result is bit-equal to the device's."""
    st = [float(v) for v in sched.tolist()]
    lr, best, bad, cool, factor, patience, threshold, min_lr, cooldown, eps = st
    current = float(loss)
    if current < best * (1.0 - threshold):
        best, bad = current, 0.0
    else:
        bad += 1
    if cool > 0:
        cool -= 1
        bad = 0.0
    if bad > patience:
        new_lr = max(lr * factor, min_lr)
        if lr - new_lr > eps:
            lr = new_lr
        cool, bad = cooldown, 0.0
    return torch.tensor([lr, best, bad, cool, factor, patience, threshold, min_lr, cooldown, eps], dtype=torch.float64)


# ---------------------------------------------------------------------------------------------- BatchNorm buffers
def bn_update_counts(preset: str) -> dict:
    """{BatchNorm prefix: running-statistics updates per training step}, read off one training forward of the CPU oracle
    with gradients enabled: 2 for a BatchNorm inside a reentrant checkpoint (the recomputation in backward moves the buffers
    again), 1 for the generic UNet's discarded center block (no gradient reaches it, so it is never recomputed)."""
    from oracle import unet_oracle as O
    cfg = O.PRESETS[preset]
    sd = O.build_state_dict(cfg, seed=0)
    size = 2 ** (cfg.n_blocks if cfg.family == "generic" else 4)
    x = torch.rand(2, cfg.input_channels, size, size, size, generator=torch.Generator().manual_seed(0))
    for k in sd:
        if not k.endswith(("running_mean", "running_var", "num_batches_tracked")):
            sd[k].requires_grad_()
    before = {k[:-len(".num_batches_tracked")]: int(v) for k, v in sd.items() if k.endswith("num_batches_tracked")}
    O.unet_forward(sd, x, cfg, training=True)
    return {k: int(sd[k + ".num_batches_tracked"]) - n for k, n in before.items()}


# ---------------------------------------------------------------------------------------------- flat gradient buffer
def slot_table(model) -> list:
    """[(parameter name, offset, numel)] of the flat gradient buffer: every trainable parameter in gradient-production
    order (the reverse of ``named_parameters()``), packed without gaps.  The generic UNet's center block (``cblock.``)
    receives no gradient and has no slice; recAE_v2_fixed and UNet4_2IC train their center block and keep it."""
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    if type(model).__name__ not in ("recAE_v2_fixed", "UNet4_2IC"):
        named = [(n, p) for n, p in named if not n.startswith("cblock.")]
    out, off = [], 0
    for n, p in reversed(named):
        out.append((n, off, p.numel()))
        off += p.numel()
    return out


# ---------------------------------------------------------------------------------------------- gradient noise floor
def oracle_grads(name: str, sd: dict, x, target, dtype=torch.float32, **emulate):
    """Parameter gradients {name: tensor or None} and loss components of one training step of the oracle at the state
    ``sd`` (copied: the caller's BatchNorm buffers do not move), on the device of ``x``.  ``emulate``: ``act_round``,
    ``grad_round``, ``weight_round`` of ``unet_forward``."""
    from oracle import unet_oracle as O
    cfg = O.PRESETS[name]
    dev = x.device
    sd = {k: (v.detach().to(dev, dtype) if v.is_floating_point() else v.detach().to(dev)).clone() for k, v in sd.items()}
    pn = [k for k in sd if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))]
    for k in pn:
        sd[k].requires_grad_()
    out = O.unet_forward(sd, x.to(dtype), cfg, training=True, **emulate)
    if isinstance(out, tuple):
        loss, comps = O.loss_double_output(out, tuple(t.to(dev, dtype) for t in target), 1.0, 1.0)
    else:
        loss, comps = O.loss_single_output(out, target.to(dev, dtype), 1.0, 1.0)
    loss.backward()
    return {k: sd[k].grad for k in pn}, {k: float(v.detach()) for k, v in comps.items()}


def rel_err(a, b) -> float:
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def noise_floor(name: str, sd: dict, x, xp, target):
    """Per-tensor bound of the bf16 product's gradients at state ``sd`` on the batch (``x``, ``target``); ``xp`` is ``x``
    perturbed by a few fp32 ulps.  Returns ({parameter: entry}, loss components of the reference; entries below).

    The reference arithmetic is fp32.  For a randomly initialised BatchNorm network the weight gradients of the deep layers
    are heavily cancelling sums over millions of voxels, so ANY bf16 evaluation is tens of percent away from fp32 per tensor
    and two equally valid bf16 evaluations are tens of percent away from EACH OTHER.  The reference is therefore the faithful
    statement of the product's arithmetic -- bf16 storage of activations and of their gradients, bf16 images of the
    convolution weights, fp32 everything else (bf16gw) -- and the bound is the distance between two such statements:

        err(product, oracle_bf16gw)  <=  1.75 * max(err(oracle_bf16gw, oracle_bf16g), err(oracle_bf16g', oracle_bf16g)) + 0.01
                                          + err(oracle_fp32, oracle_fp64)

    (err = normwise relative distance; bf16g = activations and gradients rounded, weights not; bf16g' = the same on
    ``xp``.)  The last term is the reference's OWN accumulation error: a library fp32 convolution sums the 1x1x1 head's
    bias gradient over millions of voxels in fp32 (0.57 % off its fp64 value at 128^3 on the CPU) -- the product, with
    block-wise fp32 partials, is not.  Each entry is None for a parameter without gradient, else (reference, bound,
    err(oracle_fp32, oracle_fp64)) with bound None where the gradient is analytically zero (a convolution bias in front
    of a BatchNorm: norm below 1e-6)."""
    bf = torch.bfloat16
    g16, _ = oracle_grads(name, sd, x, target, act_round=bf, grad_round=True)
    g16p, _ = oracle_grads(name, sd, xp, target, act_round=bf, grad_round=True)
    g16w, comps_w = oracle_grads(name, sd, x, target, act_round=bf, grad_round=True, weight_round=True)
    g32, _ = oracle_grads(name, sd, x, target)
    g64, _ = oracle_grads(name, sd, x, target, dtype=torch.float64)
    out = {}
    for k, ref in g16w.items():
        if ref is None:
            out[k] = None
        elif float(ref.norm()) < 1e-6:
            out[k] = (ref, None, None)
        else:
            ref_acc = rel_err(g32[k], g64[k])
            floor = max(rel_err(g16w[k], g16[k]), rel_err(g16p[k], g16[k]))
            out[k] = (ref, 1.75 * floor + 0.01 + ref_acc, ref_acc)
    return out, comps_w
