"""The BatchNorm+ReLU(+MaxPool) kernels (csrc/bn.cu) and the fused head + Dice/CE kernels (csrc/head.cu) against float64
references (norm_head_oracle.py), at every BatchNorm launch geometry of the benchmarked step (UNetSP and recAE_v2_fixed
at batch 4 x 128^3), on inputs chosen where kernels go wrong, and at the edges of their launch schedules.

Every output is held to a bound derived from the kernel's arithmetic (see the oracle's docstrings), not to a fraction of
its largest value.  The ReLU gates and pooling arg-maxes whose fp32 evaluation could go either way are classified by the
reference; either branch is accepted there and the count is reported, everywhere else the routing must be exact.
The worst ratio to each bound is printed per family."""
import collections

import pytest
import torch

import norm_head_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda"
WORST = collections.defaultdict(float)
TIES = collections.Counter()


def _note(family, r, what):
    WORST[family] = max(WORST[family], r)
    assert r <= 1.0, "%s: error at %.3f of its bound (%s)" % (family, r, what)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nworst ratio to the bound per family:")
    for k in sorted(WORST):
        print("  %-22s %.3f" % (k, WORST[k]))
    print("tie-marked decisions: %d ReLU gates, %d pooling windows" % (TIES["gate"], TIES["window"]))


# ---------------------------------------------------------------------------------------------------------------------
# (a) Every BatchNorm launch of UNetSP (c 7..112) and recAE_v2_fixed (c 8..128) at batch 4 x 128^3:
# (model, c, (n, d, h, w) of the natural volume, pooled, phase-major input, backward).  The phase-major inputs are the
# outputs of the fused up-sampling stages; c112 @ 8^3 is UNetSP's discarded center block (forward only, no tape).
MODEL_BN = [
    ("UNetSP", 7, (4, 128, 128, 128), False, False, True),
    ("UNetSP", 7, (4, 128, 128, 128), True, False, True),
    ("UNetSP", 7, (4, 128, 128, 128), False, True, True),
    ("UNetSP", 14, (4, 64, 64, 64), False, False, True),
    ("UNetSP", 14, (4, 64, 64, 64), True, False, True),
    ("UNetSP", 14, (4, 64, 64, 64), False, True, True),
    ("UNetSP", 28, (4, 32, 32, 32), False, False, True),
    ("UNetSP", 28, (4, 32, 32, 32), True, False, True),
    ("UNetSP", 28, (4, 32, 32, 32), False, True, True),
    ("UNetSP", 56, (4, 16, 16, 16), False, False, True),
    ("UNetSP", 56, (4, 16, 16, 16), True, False, True),
    ("UNetSP", 112, (4, 8, 8, 8), False, False, False),
    ("recAE", 8, (4, 128, 128, 128), False, False, True),
    ("recAE", 8, (4, 128, 128, 128), True, False, True),
    ("recAE", 8, (4, 128, 128, 128), False, True, True),
    ("recAE", 16, (4, 64, 64, 64), False, False, True),
    ("recAE", 16, (4, 64, 64, 64), True, False, True),
    ("recAE", 16, (4, 64, 64, 64), False, True, True),
    ("recAE", 32, (4, 32, 32, 32), False, False, True),
    ("recAE", 32, (4, 32, 32, 32), True, False, True),
    ("recAE", 32, (4, 32, 32, 32), False, True, True),
    ("recAE", 64, (4, 16, 16, 16), False, False, True),
    ("recAE", 64, (4, 16, 16, 16), True, False, True),
    ("recAE", 128, (4, 8, 8, 8), False, False, True),
]

# Kernel-table rows without a geometry label, and the cases that run them.
UNLABELLED = {
    "ctu_bn_finalize": "the 128^3 cases of MODEL_BN (more than BN_FOLD_MAX_VOXELS voxels)",
    "ctu_bn_running_update": "every MODEL_BN case with a backward pass (extra_updates=1)",
    "ctu_head_loss_fwd": "HEAD_CASES",
    "ctu_head_loss_bwd": "HEAD_CASES",
    "ctu_head_param_grad": "HEAD_CASES",
}


def bn_case_id(c):
    model, ch, (n, d, h, w), pool, pm, bwd = c
    return "%s-c%d@%dx%dx%dx%d%s%s%s" % (model, ch, n, d, h, w, "+pool" if pool else "", "-pm" if pm else "",
                                        "" if bwd else "-fwd")


def bn_launch_labels(case):
    """The kernel-table labels (bench.describe) of the BatchNorm launches one MODEL_BN case makes."""
    _, c, (n, d, h, w), pool, _, bwd = case
    at = "c%d @%dx%dx%dx%d" % (c, n, d, h, w)
    out = {"ctu_bn_relu_fwd %s%s" % (at, " +pool" if pool else "")}
    if bwd:
        out |= {"ctu_bn_relu_bwd_reduce %s" % at, "ctu_bn_relu_bwd_apply %s" % at}
    return out


# ---------------------------------------------------------------------------------------------------------------------
KINDS = ("typical", "shifted", "constant", "dead", "neg_gamma")


def make_bn_inputs(c, dims, seed, dtype=torch.bfloat16):
    """Natural input y [n][c][d][h][w] (stored values), gamma, beta, running stats: channel j is of kind
    KINDS[j % 5] -- typical, shifted (|mean| / std = 100), constant (var = 0), ReLU-dead everywhere, negative gamma."""
    n, d, h, w = dims
    g = torch.Generator(device=DEV).manual_seed(seed)
    y = torch.randn(n, c, d, h, w, generator=g, device=DEV) * 1.5 + 0.3
    gam = torch.rand(c, generator=g, device=DEV) + 0.5
    bet = torch.randn(c, generator=g, device=DEV) * 0.2
    for j in range(c):
        kind = KINDS[j % len(KINDS)]
        if kind == "shifted":
            y[:, j] = torch.randn(n, d, h, w, generator=g, device=DEV) + 100.0
        elif kind == "constant":
            y[:, j] = 0.75
        elif kind == "dead":
            bet[j] = -20.0 * gam[j]            # beyond 13 standard deviations: below zero at every voxel
        elif kind == "neg_gamma":
            gam[j] = -gam[j]
    y = y.to(dtype).float()
    rm = torch.randn(c, generator=g, device=DEV) * 0.1
    rv = torch.rand(c, generator=g, device=DEV) + 0.5
    return y, gam, bet, rm, rv


def _bf16(t):
    return t.to(torch.bfloat16).float()


def _pad_lanes_zero(buf, c, what, phase_major=False):
    """Lanes c..cpad-1 of the last channel block (of every phase for a phase-major tensor) are exactly 0."""
    if c % 8 == 0:
        return
    if phase_major:
        n, c8 = buf.shape[:2]
        buf = buf.reshape(n, 8, c8 // 8, *buf.shape[2:])
        pad = buf[:, :, -1, ..., c % 8:]
    else:
        pad = buf[:, -1, ..., c % 8:]
    assert int(torch.count_nonzero(pad)) == 0, "%s: pad lanes not zero" % what


def run_bn(c, dims, pool=False, pm=False, bwd=True, keep_p=None, seed=0, exact_sums=True, label=""):
    """One BatchNorm3d + ReLU (+ MaxPool3d) stage through Engine.bn_relu (extra_updates=1, as the checkpointed models
    call it) and run_tape, every output against its float64 reference and bound."""
    import ctunet_b200.engine as E
    n, D, H, W = dims
    y, gam, bet, rm0, rv0 = make_bn_inputs(c, dims, seed)
    keep = None
    if keep_p is not None:
        g = torch.Generator(device=DEV).manual_seed(seed + 7)
        cpad = (c + 7) // 8 * 8
        keep = torch.zeros(n, cpad, device=DEV)
        kept = float(torch.tensor(1.0) / (torch.tensor(1.0) - torch.tensor(keep_p)))
        keep[:, :c] = (torch.rand(n, c, generator=g, device=DEV) >= keep_p).float() * kept
        keep[:, 0] = 0.0                                         # dropped in every sample
    eng = E.Engine(torch.device(DEV), "bf16", True)
    bn = torch.nn.BatchNorm3d(c).to(DEV)
    with torch.no_grad():
        bn.weight.copy_(gam)
        bn.bias.copy_(bet)
        bn.running_mean.copy_(rm0)
        bn.running_var.copy_(rv0)
    cpad = (c + 7) // 8 * 8
    if pm:
        ya = eng.pack(O.to_phase(y))
        ya.c_nat = c
    else:
        ya = eng.pack(y)
    s, s2 = O.batch_sums(y)
    es = es2 = None
    if exact_sums:                 # what the producing convolution's epilogue hands over (checked by the conv tests)
        sums = torch.zeros(2 * cpad, dtype=torch.float64, device=DEV)
        sums[:c], sums[cpad:cpad + c] = s, s2
        ya.sums = sums
    else:                          # ctu_bn_stats computes them
        es, es2 = O.stats_sum_error(y)
    count = float(y.numel() // c)
    res = eng.bn_relu(ya, bn, True, extra_updates=1 if bwd else 0, pool=pool, keep=keep)
    a, pooled = res if pool else (res, None)
    ss = a.bn["ss"].clone()
    torch.cuda.synchronize()

    # finalisation: ss against float64
    fin = O.finalize(s, s2, count, gam, bet, bn.eps)
    dfin = O.finalize_bounds(fin, gam, bet, count, bn.eps, es, es2)
    ssk = ss.double().view(4, cpad)
    for i, key in enumerate(("scale", "shift", "mean", "invstd")):
        r, idx = O.ratio(ssk[i, :c], fin[key], dfin[key])
        _note("bn.ss." + key, r, "%s channel %d" % (label, idx))
        assert int(torch.count_nonzero(ssk[i, c:])) == 0, "ss pad lanes"
    sc, sh, mean, invstd = (ssk[i, :c] for i in range(4))

    # forward outputs from the kernel's scale / shift
    kp = keep[:, :c] if keep is not None else None
    a_ref = O.bn_forward(y, sc, sh, kp)
    a_got = eng.unpack(a)
    r, idx = O.ratio(a_got, a_ref, O.act_bound(a_ref, torch.bfloat16, kp))
    _note("bn.a", r, "%s flat %d" % (label, idx))
    _pad_lanes_zero(a.buf, c, "a")
    if pool:
        p_ref = O.pool_forward(a_ref)
        r, idx = O.ratio(eng.unpack(pooled), p_ref, O.act_bound(p_ref, torch.bfloat16, kp))
        _note("bn.pooled", r, "%s flat %d" % (label, idx))
        _pad_lanes_zero(pooled.buf, c, "pooled")

    updates = 2 if bwd else 1
    if not bwd:
        rm, rv = O.running(rm0, rv0, fin, count, bn.momentum, updates)
        em, ev = O.running_bounds(rm0, rv0, fin, dfin, count, bn.momentum, updates)
        _note("bn.running", max(O.ratio(bn.running_mean, rm, em)[0], O.ratio(bn.running_var, rv, ev)[0]), label)
        assert int(bn.num_batches_tracked) == 1
        return

    # backward
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    dA = _bf16(torch.randn(n, c, D, H, W, generator=g, device=DEV))
    dP = _bf16(torch.randn(n, c, D // 2, H // 2, W // 2, generator=g, device=DEV) * 2) if pool else None
    eng.agrads[id(a)] = eng.pack(dA)
    if pool:
        eng.agrads[id(pooled)] = eng.pack(dP)
    eng.run_tape()
    torch.cuda.synchronize()
    dy_act = eng.agrads[id(ya)]
    dy = eng.unpack(dy_act)
    if pm:
        dy = O.from_phase(dy, c)
    _pad_lanes_zero(dy_act.buf, c, "dy", phase_major=pm)
    dg, db = eng.pgrads[id(bn.weight)], eng.pgrads[id(bn.bias)]

    ss4 = (sc, sh, mean, invstd)
    ref, err, gate_tie, route_tie = O.dy_error_with_ties(y, ss4, dA, dP, kp, dy)
    TIES["gate"] += int(gate_tie.sum())
    if pool:
        TIES["window"] += int(route_tie.sum())
    # the gradient a tied decision may send elsewhere: |dA| at a tied gate, |dP| over the children of a tied window
    tie_dz = torch.where(gate_tie, dA.double(), torch.zeros_like(ref["dz"]))
    if pool:
        tie_dz = tie_dz + O.unwindows(route_tie.unsqueeze(-1).double().expand(*route_tie.shape, 8) * dP.double().unsqueeze(-1))
    if kp is not None:
        tie_dz = tie_dz * kp.double()[:, :, None, None, None]
    mode = O.bn_mode(pool, pm, D, H, W)
    bnd = O.bn_backward_bounds(ref, ss4, O.reduce_depth(mode, n, c, D, H, W), torch.bfloat16, tie_dz)
    r, idx = O.ratio(err, torch.zeros_like(err), bnd["dy"])
    _note("bn.dy", r, "%s flat %d" % (label, idx))
    r, idx = O.ratio(db, ref["dbeta"], bnd["dbeta"])
    _note("bn.dbeta (sum dz)", r, "%s channel %d" % (label, idx))
    r, idx = O.ratio(dg, ref["dgamma"], bnd["dgamma"])
    _note("bn.dgamma (sum dz xhat)", r, "%s channel %d" % (label, idx))
    if kp is not None:
        assert float(dy[:, 0].abs().max()) == 0.0 and float(dg[0]) == 0.0 and float(db[0]) == 0.0

    rm, rv = O.running(rm0, rv0, fin, count, bn.momentum, updates)
    em, ev = O.running_bounds(rm0, rv0, fin, dfin, count, bn.momentum, updates)
    _note("bn.running", max(O.ratio(bn.running_mean, rm, em)[0], O.ratio(bn.running_var, rv, ev)[0]), label)
    assert int(bn.num_batches_tracked) == 2


@pytest.mark.parametrize("case", MODEL_BN, ids=bn_case_id)
def test_bn_model_launches(case):
    _, c, dims, pool, pm, bwd = case
    run_bn(c, dims, pool=pool, pm=pm, bwd=bwd, seed=c, label=bn_case_id(case))


# (c) Edges: (c, (n, d, h, w), pool, phase-major, keep p, exact sums)
EDGE_BN = [
    (9, (2, 9, 5, 7), False, False, None, True),          # odd dims: mode 0 (one voxel per thread); c = 9: one lane in block 2
    (9, (2, 9, 5, 7), False, False, 0.3, True),           # dropout, mode 0
    (7, (2, 16, 12, 20), True, False, 0.3, True),         # dropout, mode 1 (pooled)
    (12, (3, 10, 14, 22), False, False, 0.5, False),      # dropout, mode 3; 3080 voxels: not a multiple of 8192 / 2048
    (9, (4, 64, 64, 62), True, False, None, True),        # just below BN_FOLD_MAX_VOXELS (folded finalisation)
    (9, (4, 64, 64, 64), False, True, None, True),        # exactly on it (folded, <=)
    (9, (4, 64, 64, 66), False, False, None, True),       # just above it (ctu_bn_finalize)
    (7, (1, 32, 48, 40), True, False, None, True),        # n = 1
    (9, (2, 10, 6, 14), False, True, None, False),        # phase-major, stats from ctu_bn_stats, 840 voxels
    (7, (3, 6, 10, 14), True, False, None, False),        # pooled, ctu_bn_stats
]


@pytest.mark.parametrize("case", EDGE_BN, ids=lambda c: "c%d@%dx%dx%dx%d%s%s%s%s" % (
    c[0], *c[1], "+pool" if c[2] else "", "-pm" if c[3] else "", "-drop" if c[4] else "", "" if c[5] else "-stats"))
def test_bn_edges(case):
    c, dims, pool, pm, keep_p, exact = case
    run_bn(c, dims, pool=pool, pm=pm, keep_p=keep_p, seed=100 + c, exact_sums=exact, label=str(case))


# ---------------------------------------------------------------------------------------------------------------------
# (d) Fused head + loss: (name, flags, source channels, cout, (n, d, h, w), uint8 targets, (ce_l, dice_l))
F_SP = O.HEAD_SIGMOID | O.HEAD_SP
F_SPS = O.HEAD_SIGMOID | O.HEAD_SP_SOFTMAX
HEAD_CASES = [
    ("UNetSP-u8", F_SP, [7, 7], 3, (4, 128, 128, 128), True, (1.0, 1.0)),
    ("UNetSP-onehot", F_SP, [7, 7], 3, (4, 128, 128, 128), False, (1.0, 1.0)),
    ("recAE-u8", O.HEAD_SOFTMAX, [8, 8], 2, (4, 128, 128, 128), True, (1.0, 1.0)),
    ("UNetSPSmall", F_SPS, [4, 4], 3, (2, 64, 64, 64), False, (1.0, 0.0)),
    ("UNetSP-dice2", F_SP, [7, 7], 3, (2, 48, 40, 36), True, (0.0, 2.0)),
    ("odd-SP", F_SP, [7], 3, (3, 31, 33, 35), True, (1.0, 1.0)),
    ("odd-plain", O.HEAD_SOFTMAX, [8, 8], 2, (3, 31, 33, 35), False, (0.0, 2.0)),
    ("n1-SP", F_SP, [7, 7], 3, (1, 128, 128, 128), True, (1.0, 1.0)),
    ("n7-plain", O.HEAD_SOFTMAX, [8, 8], 2, (7, 64, 64, 48), False, (1.0, 0.0)),
]


def run_head(name, flags, chans, cout, dims, u8, weights, seed=0):
    import ctunet_b200.engine as E
    from ctunet_b200 import _lib as L
    from oracle import unet_oracle as UO
    n, d, h, w = dims
    spatial = d * h * w
    sp = bool(flags & (O.HEAD_SP | O.HEAD_SP_SOFTMAX))
    ce_l, dice_l = weights
    sfd = sp                                   # the double-output handler takes Dice on softmax(pred), the single one not
    g = torch.Generator(device=DEV).manual_seed(seed)
    xs = [_bf16(torch.relu(torch.randn(n, c, d, h, w, generator=g, device=DEV) * 1.2 + 0.2)) for c in chans]
    cin = sum(chans)
    W = torch.randn(cout, cin, generator=g, device=DEV) * 0.5
    b = torch.randn(cout, generator=g, device=DEV) * 0.1
    x = torch.cat(xs, 1)
    lc = O.head_logits(x, W, b)
    # targets correlated with the logits (the loss then has signal in every term), with noise
    noise = torch.randn(n, d, h, w, generator=g, device=DEV)
    masks = [(lc[:, 0] + 0.5 * noise > lc[:, 0].median()).to(torch.uint8)]
    if sp:
        masks.append((lc[:, 1] - 0.5 * noise > lc[:, 1].median()).to(torch.uint8))
    tgts64 = [O.onehot_targets(m, True) for m in masks]
    if cout > 2 and not sp:
        raise AssertionError("plain cases use two classes")
    targets = [m.contiguous() if u8 else t.float().contiguous() for m, t in zip(masks, tgts64)]
    pairs = len(targets)

    eng = E.Engine(torch.device(DEV), "bf16", True)
    srcs = [eng.pack(t) for t in xs]
    pa, ca, ns = eng._src_args(srcs)
    t0, t1 = targets[0].data_ptr(), (targets[1].data_ptr() if sp else None)
    sums = torch.empty(4 * pairs * n, dtype=torch.float64, device=DEV)
    ncomp = pairs * ((ce_l != 0) + (dice_l != 0)) + 1
    comps = torch.empty(ncomp, dtype=torch.float32, device=DEV)
    st = L.stream_ptr()
    L.call("ctu_head_loss_fwd", eng.dtype, pa, ca, ns, W.data_ptr(), b.data_ptr(), cout, flags, t0, t1, int(u8), int(sfd),
           float(ce_l), float(dice_l), sums.data_ptr(), comps.data_ptr(), None, n, spatial, st)
    dsrcs = [eng.new_act(s.c, s.n, s.d, s.h, s.w) for s in srcs]
    dlc = torch.empty(n, cout, d, h, w, dtype=torch.float32, device=DEV)
    L.call("ctu_head_loss_bwd", eng.dtype, pa, ca, ns, W.data_ptr(), b.data_ptr(), cout, flags, t0, t1, int(u8), int(sfd),
           float(ce_l), float(dice_l), sums.data_ptr(), L.ptr_array([s.ptr for s in dsrcs]), dlc.data_ptr(), n, spatial, st)
    dW = torch.empty(cout, cin, device=DEV)
    db = torch.empty(cout, device=DEV)
    L.call("ctu_head_param_grad", eng.dtype, pa, ca, ns, dlc.data_ptr(), cout, dW.data_ptr(), db.data_ptr(), n, spatial, st)
    torch.cuda.synchronize()

    # per-sample sums and components
    preds = O.head_chain(lc, flags)
    lc_err = O.logit_error(x, W, b)
    eps_pred = O.chain_error(lc, lc_err)
    ref_sums = torch.stack([O.pair_sums(p, t, sfd) for p, t in zip(preds, tgts64)])
    depth = O.head_loss_depth(n, spatial, 2)
    dsums = torch.stack([O.loss_sums_bounds(p, t, sfd, eps_pred, depth) for p, t in zip(preds, tgts64)])
    if not ce_l:                                  # CrossEntropy off: the kernels leave its sum at 0
        ref_sums[..., 3] = 0.0
        dsums[..., 3] = 0.0
    ks = sums.view(pairs, n, 4)
    r, idx = O.ratio(ks, ref_sums, dsums)
    _note("head.sums", r, "%s flat %d" % (name, idx))
    if sp:
        _, cd = UO.loss_double_output(preds, tgts64, dice_l, ce_l)
    else:
        _, cd = UO.loss_single_output(preds[0], tgts64[0], dice_l, ce_l)
    ref_comps = torch.stack([cd[k].double() for k in cd])
    r, idx = O.ratio(comps, ref_comps, O.components_bounds(ref_sums, dsums, spatial, ce_l, dice_l))
    _note("head.components", r, "%s component %d" % (name, idx))

    # logit gradients from the kernel's sums, then everything downstream from the kernel's dlc
    ref_dlc = O.logit_gradients(lc, flags, tgts64, ks, sfd, ce_l, dice_l, spatial)
    kce = ce_l / (n * spatial) if ce_l else 0.0
    bnd = O.dlc_bounds(O.dice_coefficients(ks, n, dice_l), kce, eps_pred, lc_err.amax(1), n)
    r, idx = O.ratio(dlc, ref_dlc, bnd.expand_as(ref_dlc))
    _note("head.dlc", r, "%s flat %d" % (name, idx))
    ref_dsrc, bnd = O.dsrc_ref_and_bound(dlc, W, torch.bfloat16)
    got = torch.cat([eng.unpack(s) for s in dsrcs], 1)
    r, idx = O.ratio(got, ref_dsrc, bnd)
    _note("head.dsrc", r, "%s flat %d" % (name, idx))
    for s, c in zip(dsrcs, chans):
        _pad_lanes_zero(s.buf, c, "dsrc")
    rw, rb, bw, bb = O.param_grad_ref_and_bound(dlc, x, O.param_grad_depth(n, spatial, sum((c + 7) // 8 for c in chans)))
    r, idx = O.ratio(dW, rw, bw)
    _note("head.dW", r, "%s flat %d" % (name, idx))
    r, idx = O.ratio(db, rb, bb)
    _note("head.db", r, "%s flat %d" % (name, idx))


@pytest.mark.parametrize("case", HEAD_CASES, ids=lambda c: c[0])
def test_head_loss(case):
    run_head(*case)
