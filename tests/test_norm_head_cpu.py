"""The float64 references and bounds of tests/test_gpu_norm_head.py checked on the CPU: the references against autograd of
torch's own BatchNorm3d -> relu -> max_pool3d and of the reference loss, a float32 emulation of the kernels' formulas
inside every bound, perturbations the size of a real defect outside it, the case table against the profiled launches, and
the alignment checks of the fused head + loss and the loss entry points (which return before any CUDA call)."""
import os
import re
import types

import pytest
import torch
import torch.nn.functional as F

import norm_head_oracle as O
import test_gpu_norm_head as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROFILE_TABLES = ["profiles/r2_kernel_table_g_UNetSP.txt", "profiles/r2_kernel_table_e_recAE.txt"]
EPS = 1e-5


def _inputs(c, dims, seed, kinds=True):
    """CPU version of the GPU test's inputs: bf16-stored y with one channel of each kind."""
    n, d, h, w = dims
    g = torch.Generator().manual_seed(seed)
    y = torch.randn(n, c, d, h, w, generator=g) * 1.5 + 0.3
    gam = torch.rand(c, generator=g) + 0.5
    bet = torch.randn(c, generator=g) * 0.2
    for j in range(c if kinds else 0):
        kind = T.KINDS[j % len(T.KINDS)]
        if kind == "shifted":
            y[:, j] = torch.randn(n, d, h, w, generator=g) + 100.0
        elif kind == "constant":
            y[:, j] = 0.75
        elif kind == "dead":
            bet[j] = -20.0 * gam[j]
        elif kind == "neg_gamma":
            gam[j] = -gam[j]
    y = y.to(torch.bfloat16).float()
    dA = torch.randn(n, c, d, h, w, generator=g).to(torch.bfloat16).float()
    dP = (torch.randn(n, c, d // 2, h // 2, w // 2, generator=g) * 2).to(torch.bfloat16).float()
    return y, gam, bet, dA, dP, g


# ---------------------------------------------------------------------------------------------------------------------
# the references against autograd
@pytest.mark.parametrize("pool", [False, True])
@pytest.mark.parametrize("drop", [False, True])
def test_bn_reference_matches_autograd(pool, drop):
    c, dims = 7, (2, 4, 6, 8)
    y, gam, bet, dA, dP, g = _inputs(c, dims, 1, kinds=False)
    keep = ((torch.rand(2, c, generator=g) > 0.3).double() / 0.7) if drop else None
    yd = y.double().requires_grad_()
    gd, bd = gam.double().requires_grad_(), bet.double().requires_grad_()
    rm, rv = torch.zeros(c, dtype=torch.float64), torch.ones(c, dtype=torch.float64)
    a = F.relu(F.batch_norm(yd, rm, rv, gd, bd, True, 0.1, EPS))
    if drop:
        a = a * keep[:, :, None, None, None]
    outs, grads = [a], [dA.double()]
    if pool:
        outs.append(F.max_pool3d(a, 2, 2))
        grads.append(dP.double())
    torch.autograd.backward(outs, grads)

    s, s2 = O.batch_sums(y)
    count = y.numel() / c
    fin = O.finalize(s, s2, count, gam, bet, EPS)
    a_ref = O.bn_forward(y, fin["scale"], fin["shift"], keep)
    assert torch.allclose(a_ref, outs[0].detach(), rtol=1e-12, atol=1e-12)
    if pool:
        assert torch.allclose(O.pool_forward(a_ref), outs[1].detach(), rtol=1e-12, atol=1e-12)
    ss = (fin["scale"], fin["shift"], fin["mean"], fin["invstd"])
    ref = O.bn_backward(y, ss, dA, dP if pool else None, keep)
    assert torch.allclose(ref["dy"], yd.grad, rtol=1e-9, atol=1e-11)
    assert torch.allclose(ref["dgamma"], gd.grad, rtol=1e-10, atol=1e-11)
    assert torch.allclose(ref["dbeta"], bd.grad, rtol=1e-10, atol=1e-11)
    # running statistics: torch's update, twice (the forward and the checkpoint's recomputation)
    bn = torch.nn.BatchNorm3d(c).double()
    rm0, rv0 = torch.randn(c, generator=g) * 0.1, torch.rand(c, generator=g) + 0.5
    with torch.no_grad():
        bn.running_mean.copy_(rm0)
        bn.running_var.copy_(rv0)
        bn.momentum = float(torch.tensor(0.1, dtype=torch.float32))
        bn(y.double())
        bn(y.double())
    erm, erv = O.running(rm0, rv0, fin, count, 0.1, 2)
    assert torch.allclose(erm, bn.running_mean, rtol=1e-12, atol=1e-14)
    assert torch.allclose(erv, bn.running_var, rtol=1e-12, atol=1e-14)


def test_phase_layout_round_trip_and_windows():
    x = torch.randn(2, 9, 4, 6, 8, dtype=torch.float64)
    ph = O.to_phase(x)
    assert ph.shape == (2, 8 * 16, 2, 3, 4)
    assert torch.equal(O.from_phase(ph, 9), x)
    assert torch.equal(O.unwindows(O.windows(x)), x)
    # window child q = qd*4 + qh*2 + qw is phase block q
    q = 5
    assert torch.equal(O.windows(x)[..., q], ph.view(2, 8, 16, 2, 3, 4)[:, q, :9])
    # the first maximum wins, as torch.max_pool3d routes its gradient
    v = torch.zeros(1, 1, 2, 2, 2, dtype=torch.float64)
    v[0, 0, 1, 0, 1] = 3.0
    v[0, 0, 1, 1, 1] = 3.0
    win, tie = O.window_winners(v)
    assert int(win) == 5 and not bool(tie)


@pytest.mark.parametrize("flags,sp", [(T.F_SP, True), (T.F_SPS, True), (O.HEAD_SOFTMAX, False), (0, False)])
@pytest.mark.parametrize("weights", [(1.0, 1.0), (1.0, 0.0), (0.0, 2.0)])
def test_head_reference_matches_oracle_loss(flags, sp, weights, monkeypatch):
    """Sums, components and logit gradients of the head references against autograd of oracle.unet_oracle's loss."""
    from oracle import unet_oracle as UO
    ce_l, dice_l = weights
    g = torch.Generator().manual_seed(7)
    n, cout, cin, dims = 2, (3 if sp else 2), 9, (3, 4, 5)
    x = torch.relu(torch.randn(n, cin, *dims, generator=g, dtype=torch.float64))
    w = torch.randn(cout, cin, generator=g, dtype=torch.float64) * 0.5
    b = torch.randn(cout, generator=g, dtype=torch.float64) * 0.1
    lc = O.head_logits(x, w, b).requires_grad_()
    masks = [(torch.rand(n, *dims, generator=g) > 0.5).to(torch.uint8) for _ in range(2 if sp else 1)]
    tgts = [O.onehot_targets(m, True) for m in masks]
    preds = O.head_chain(lc, flags)
    if sp:
        total, comps = UO.loss_double_output(preds, tgts, dice_l, ce_l)
    else:
        total, comps = UO.loss_single_output(preds[0], tgts[0], dice_l, ce_l)
    (g_ref,) = torch.autograd.grad(total, lc)
    spatial = 60
    sums = torch.stack([O.pair_sums(p.detach(), t, sp) for p, t in zip(preds, tgts)])
    assert torch.allclose(O.components(sums, spatial, ce_l, dice_l), torch.stack([v.detach() for v in comps.values()]),
                          rtol=1e-12, atol=1e-14)
    # exact (float64) Dice coefficients: the surrogate's gradient is the loss's gradient
    monkeypatch.setattr(O, "fp32", lambda t: t)
    dlc = O.logit_gradients(lc.detach(), flags, tgts, sums, sp, ce_l, dice_l, spatial)
    assert torch.allclose(dlc, g_ref, rtol=1e-10, atol=1e-14)


# ---------------------------------------------------------------------------------------------------------------------
# the bounds are tight: the kernels' formulas in float32 sit inside, a defect-sized perturbation does not
def _f(t):
    return t.float().double()


def _emulate(y, gam, bet, dA, dP, pool):
    """bn.cu's arithmetic in float32 (fmaf as one rounding of the float64 value), with bf16 outputs."""
    c = y.shape[1]
    s, s2 = O.batch_sums(y)
    count = y.numel() / c
    mean = s / count
    var = (s2 / count - mean * mean).clamp_min(0)
    invstd = _f(1.0 / torch.sqrt(var + EPS))
    meanf = _f(mean)
    scale = _f(gam.double() * invstd)
    shift = _f(bet.double() - _f(meanf * scale))
    ch = O._ch
    av = _f(y.double() * ch(scale) + ch(shift))
    a = _f(av.clamp_min(0)).to(torch.bfloat16).double()
    win = O.window_winners(O.preact(y, scale, shift))[0] if pool else None
    gsum = dA.double()
    if pool:
        onehot = F.one_hot(win, 8).double()
        gsum = _f(gsum + O.unwindows(onehot * dP.double().unsqueeze(-1)))
    dz = torch.where(av > 0, gsum, torch.zeros_like(gsum))
    xhat = _f(_f(y.double() - ch(meanf)) * ch(invstd))
    s1 = _f(dz).float().sum((0, 2, 3, 4)).double()
    s2b = _f(dz * xhat).float().sum((0, 2, 3, 4)).double()
    k1, k2 = _f(s1 / count), _f(s2b / count)
    o = _f(ch(scale) * _f(_f(dz - ch(k1)) - _f(xhat * ch(k2))))
    dy = o.to(torch.bfloat16).double()
    return dict(scale=scale, shift=shift, mean=meanf, invstd=invstd, a=a, dy=dy, dbeta=_f(s1), dgamma=_f(s2b),
                fin=O.finalize(s, s2, count, gam, bet, EPS), count=count)


@pytest.mark.parametrize("pool", [False, True])
def test_float32_emulation_sits_inside_the_bounds_and_defects_do_not(pool):
    c, dims = 9, (2, 8, 6, 10)
    y, gam, bet, dA, dP, _ = _inputs(c, dims, 3)
    dP = dP if pool else None
    em = _emulate(y, gam, bet, dA, dP, pool)
    fin, count = em["fin"], em["count"]
    dfin = O.finalize_bounds(fin, gam, bet, count, EPS)
    for key in ("scale", "shift", "mean", "invstd"):
        assert O.ratio(em[key], fin[key], dfin[key])[0] <= 1.0, key
    ss = (em["scale"], em["shift"], em["mean"], em["invstd"])
    a_ref = O.bn_forward(y, em["scale"], em["shift"])
    abound = O.act_bound(a_ref, torch.bfloat16)
    assert O.ratio(em["a"], a_ref, abound)[0] <= 1.0
    v = O.preact(y, em["scale"], em["shift"])
    win, tie = O.window_winners(v) if pool else (None, None)
    ref = O.bn_backward(y, ss, dA, dP, None, win)
    n, _, d, h, w = y.shape
    bnd = O.bn_backward_bounds(ref, ss, O.reduce_depth(O.bn_mode(pool, False, d, h, w), n, c, d, h, w), torch.bfloat16)
    r_dy = O.ratio(em["dy"], ref["dy"], bnd["dy"])[0]
    assert r_dy <= 1.0
    assert O.ratio(em["dbeta"], ref["dbeta"], bnd["dbeta"])[0] <= 1.0
    assert O.ratio(em["dgamma"], ref["dgamma"], bnd["dgamma"])[0] <= 1.0
    # the bounds are not vacuous
    assert 0.05 < r_dy, "the dy bound is loose by more than 20x on a float32 emulation (%.3f)" % r_dy

    # one dy element off by 2 bf16 ulps
    bad = em["dy"].clone().reshape(-1)
    i = int(bad.abs().argmax())
    bad[i] += 2 * 2.0 ** (torch.floor(torch.log2(bad[i].abs())) - 7)
    assert O.ratio(bad.view_as(em["dy"]), ref["dy"], bnd["dy"])[0] > 1.0

    # one channel's scale off by 2^-7
    sc_bad = em["scale"].clone()
    sc_bad[0] *= 1 + 2.0 ** -7
    assert O.ratio(sc_bad, fin["scale"], dfin["scale"])[0] > 1.0
    assert O.ratio(O.bn_forward(y, sc_bad, em["shift"]), a_ref, abound)[0] > 1.0

    if pool:
        # one window routed to its runner-up: pick an untied window of the typical channel with every gate open
        assert not bool(tie.any())
        r = O.windows(v.clamp_min(0))
        ok = ((r > 0).sum(-1) >= 2) & (dP.double().abs() > 0.5)      # winner and runner-up both pass the gate
        idx = ok[:, 0].nonzero()[0]
        flip = torch.zeros_like(tie)
        flip[idx[0], 0, idx[1], idx[2], idx[3]] = True
        wrong = O.bn_backward(y, ss, dA, dP, None, win, flip_route=flip)
        assert O.ratio(wrong["dy"].to(torch.bfloat16).double(), ref["dy"], bnd["dy"])[0] > 1.0


def test_head_bounds_hold_for_float32_and_catch_truncated_source_gradients():
    """dsrc from the kernel's dlc: round-to-nearest bf16 of the fp32 fmaf chain sits inside; rounding toward zero does
    not.  dW / db: an fp32 sum inside, the loss of one block's atomics (of 296) outside."""
    g = torch.Generator().manual_seed(11)
    n, cout, cin, sp = 2, 3, 14, 4096
    dlc = (torch.randn(n, cout, sp, generator=g) * 1e-4).float()
    w = torch.randn(cout, cin, generator=g) * 0.5
    ref, bnd = O.dsrc_ref_and_bound(dlc, w, torch.bfloat16)
    f32 = torch.einsum("no...,oc->nc...", dlc, w)
    assert O.ratio(f32.to(torch.bfloat16), ref, bnd)[0] <= 1.0
    bits = f32.view(torch.int32) & ~0xFFFF                              # bf16 by truncation (toward zero)
    assert O.ratio(bits.view(torch.float32), ref, bnd)[0] > 1.0
    x = torch.relu(torch.randn(n, cin, sp, generator=g)).to(torch.bfloat16).float()
    dlc = dlc - 2e-5                                                     # a gradient with a sign (no cancellation)
    rw, rb, bw, bb = O.param_grad_ref_and_bound(dlc, x, O.param_grad_depth(4, 128 ** 3, 2))
    assert O.ratio(torch.einsum("nos,ncs->oc", dlc, x), rw, bw)[0] <= 1.0
    assert O.ratio(dlc.sum((0, 2)), rb, bb)[0] <= 1.0
    assert O.ratio(rb * (1 - 1 / 296), rb, bb)[0] > 1.0


# ---------------------------------------------------------------------------------------------------------------------
def test_case_table_covers_the_profiled_launches():
    """Every ctu_bn_relu_fwd / _bwd_reduce / _bwd_apply row of the benchmarked step's kernel tables is a launch of a
    MODEL_BN case, and every unlabelled BatchNorm / head row is named by a case."""
    covered = set().union(*(T.bn_launch_labels(c) for c in T.MODEL_BN))
    rows, unlabelled = [], set()
    for name in PROFILE_TABLES:
        with open(os.path.join(ROOT, name)) as f:
            for line in f:
                m = re.match(r"(ctu_bn_relu_(?:fwd|bwd_reduce|bwd_apply) c\d+ @\S+(?: \+pool)?)", line)
                if m:
                    rows.append(m.group(1))
                m = re.match(r"(ctu_(?:bn|head)_\w+)\s+\d", line)
                if m:
                    unlabelled.add(m.group(1))
    assert len(rows) >= 30
    missing = [r for r in rows if r not in covered]
    assert not missing, missing
    assert unlabelled == set(T.UNLABELLED), unlabelled ^ set(T.UNLABELLED)
    # the folded / separate finalisation boundary is exercised on both sides and exactly on it
    from ctunet_b200.engine import BN_FOLD_MAX_VOXELS
    vox = {c[1][0] * c[1][1] * c[1][2] * c[1][3] for c in T.EDGE_BN}
    assert BN_FOLD_MAX_VOXELS in vox
    assert any(0.9 * BN_FOLD_MAX_VOXELS < v < BN_FOLD_MAX_VOXELS for v in vox)
    assert any(BN_FOLD_MAX_VOXELS < v < 1.1 * BN_FOLD_MAX_VOXELS for v in vox)
    # the head grid caps: n = 1 and n = 7 both reach ceil(2368 / n) blocks per sample, and an odd voxel count
    caps = {c[4][0] for c in T.HEAD_CASES
            if O.cdiv(c[4][1] * c[4][2] * c[4][3] // 2, O.HEAD_THREADS) > O.cdiv(O.HEAD_LOSS_CAP, c[4][0])}
    assert {1, 7} <= caps
    assert any((c[4][1] * c[4][2] * c[4][3]) % 2 for c in T.HEAD_CASES)


# ---------------------------------------------------------------------------------------------------------------------
# alignment of the targets (and of the loss kernels' vector operands): refused before any memset or launch
@pytest.fixture(scope="module")
def lib():
    from ctunet_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib


def _head_loss_args(L, which, t0, t1, u8, flags=None, dlogits=0x7000):
    flags = T.F_SP if flags is None else flags
    srcs, chans = L.ptr_array([0x100000]), L.int_array([7])
    head = (L.CTU_BF16, srcs, chans, 1, 0x200000, 0x300000, 3, flags, t0, t1, u8, 1, 1.0, 1.0, 0x400000)
    if which == "fwd":
        return head + (0x500000, None, 2, 64, None)
    return head + (L.ptr_array([0x600000]), dlogits, 2, 64, None)


@pytest.mark.parametrize("which", ["fwd", "bwd"])
def test_head_loss_entries_refuse_misaligned_targets(lib, which):
    L = lib
    name = "ctu_head_loss_" + which
    with pytest.raises(RuntimeError, match="uint8 targets must be 2-byte aligned"):
        L.call(name, *_head_loss_args(L, which, 0x800001, 0x900000, 1))
    with pytest.raises(RuntimeError, match="uint8 targets must be 2-byte aligned"):
        L.call(name, *_head_loss_args(L, which, 0x800000, 0x900003, 1))
    with pytest.raises(RuntimeError, match="float32 targets must be 8-byte aligned"):
        L.call(name, *_head_loss_args(L, which, 0x800004, 0x900000, 0))
    if which == "bwd":
        with pytest.raises(RuntimeError, match="dlogits must be 8-byte aligned"):
            L.call(name, *_head_loss_args(L, which, 0x800000, 0x900000, 1, dlogits=0x7004))


def test_loss_entries_refuse_misaligned_vector_operands(lib):
    L = lib
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        L.call("ctu_dice_ce_fwd", 0x100004, 0x200000, 2, 2, 64, 1, 1, 0x300000, 0x400000, None)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        L.call("ctu_dice_ce_fwd", 0x100000, 0x200008, 2, 2, 64, 1, 1, 0x300000, 0x400000, None)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        L.call("ctu_dice_ce_bwd", 0x100000, 0x200000, 2, 2, 64, 1, 1, 0x300000, 0x400000, 0x500004, None)


@pytest.mark.parametrize("u8", [True, False])
def test_engine_head_loss_refuses_misaligned_target_views(u8):
    from ctunet_b200.engine import Act, Engine
    n, d, h, w = 2, 4, 4, 6
    s0 = Act(torch.zeros(n, 1, d, h, w, 8, dtype=torch.bfloat16), 7, n, d, h, w)
    shape = (n, d, h, w) if u8 else (n, 2, d, h, w)
    numel = n * d * h * w * (1 if u8 else 2)
    flat = torch.zeros(numel + 1, dtype=torch.uint8 if u8 else torch.float32)
    good = flat[:numel].view(shape)
    bad = flat[1:].view(shape)                       # contiguous, 1 byte (uint8) / 4 bytes (float) off
    assert bad.is_contiguous()
    fake = types.SimpleNamespace(fused_loss=([good, bad], True, 1.0, 1.0, None, None))
    with pytest.raises(TypeError, match="byte aligned"):
        Engine._head_loss(fake, [s0], torch.zeros(3, 7), torch.zeros(3), T.F_SP, True)
