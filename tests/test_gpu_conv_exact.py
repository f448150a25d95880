"""Bit-exact tests of the convolutions (conv_tc.cu, conv_wide.cu, the fused up-sampling stage of fuse.cu, the CUDA-core
kernels) on small-integer operands (conv_exact_oracle.py), at the launch geometries of the benchmarked step and at the
edges of the kernels' schedules.  A kernel that drops, duplicates or misplaces one product fails, and the failure names
the voxel, its 16 x 16 tile and its d-plane."""
import os
import re

import pytest
import torch
import torch.nn as nn

import conv_exact_oracle as X

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

# ---------------------------------------------------------------------------------------------------------------------
# (a) Every convolution of UNetSP and recAE_v2_fixed at batch 4 x 128^3, at its true shape.
# (kind, k, source channels, cout, bias, (n, d, h, w), forward variant, data-gradient variant per source, weight-gradient
# variant).  Variants: 1 conv_tc.cu, 2 conv_wide.cu (forward / data gradient) or the tap-stationary kernel (weight
# gradient).  "up": the fused ConvTranspose3d(2, 2) -> Conv3d stage, dims of its LOW-resolution input, variants of the
# composed 3^3 convolution.  "conv_fwd": forward only (the dead branch runs without a tape).
LAYERS = [
    # UNetSP (3^3, no bias)
    ("conv", 3, [2], 7, False, (4, 128, 128, 128), 1, [1], 1),         # d_blocks.0.block.0 (input gradient: 7->2)
    ("conv", 3, [7], 7, False, (4, 128, 128, 128), 1, [1], 1),         # d_blocks.0.block.3, u_blocks.3.block.4
    ("conv", 3, [7], 14, False, (4, 64, 64, 64), 1, [1], 1),           # d_blocks.1.block.0
    ("conv", 3, [14], 14, False, (4, 64, 64, 64), 1, [1], 1),          # d_blocks.1.block.3, u_blocks.2.block.4
    ("conv", 3, [14], 28, False, (4, 32, 32, 32), 1, [1], 1),          # d_blocks.2.block.0
    ("conv", 3, [28], 28, False, (4, 32, 32, 32), 1, [1], 1),          # d_blocks.2.block.3, u_blocks.1.block.4
    ("conv", 3, [28], 56, False, (4, 16, 16, 16), 2, [2], 2),          # d_blocks.3.block.0
    ("conv", 3, [56], 56, False, (4, 16, 16, 16), 2, [2], 2),          # d_blocks.3.block.3, u_blocks.0.block.1 / .4
    ("conv_fwd", 3, [56], 112, False, (4, 8, 8, 8), 2, [], 0),         # cblock.block.0 (dead branch)
    ("conv_fwd", 3, [112], 112, False, (4, 8, 8, 8), 2, [], 0),        # cblock.block.3 (dead branch)
    ("convt2", 2, [56], 56, True, (4, 8, 8, 8), 0, [0], 0),            # u_blocks.0.block.0 (8^3: not fusable)
    ("up", 3, [56, 56], 28, False, (4, 16, 16, 16), 1, [2, 2], 1),     # u_blocks.1.block.0 + .1 (dgrad 256->56)
    ("up", 3, [28, 28], 14, False, (4, 32, 32, 32), 1, [1, 1], 1),     # u_blocks.2.block.0 + .1 (dgrad 128->28)
    ("up", 3, [14, 14], 7, False, (4, 64, 64, 64), 1, [1, 1], 1),      # u_blocks.3.block.0 + .1 (dgrad 64->14)
    # recAE_v2_fixed (5^3, bias)
    ("conv", 5, [1], 8, True, (4, 128, 128, 128), 1, [1], 1),          # dblock1.0 (input gradient: 8->1)
    ("conv", 5, [8], 8, True, (4, 128, 128, 128), 1, [1], 1),          # dblock1.3, ublock4.4
    ("conv", 5, [8], 16, True, (4, 64, 64, 64), 1, [1], 1),            # dblock2.0
    ("conv", 5, [16], 16, True, (4, 64, 64, 64), 1, [1], 1),           # dblock2.3, ublock3.4
    ("conv", 5, [16], 32, True, (4, 32, 32, 32), 1, [1], 1),           # dblock3.0
    ("conv", 5, [32], 32, True, (4, 32, 32, 32), 1, [1], 1),           # dblock3.3, ublock2.4
    ("conv", 5, [32], 64, True, (4, 16, 16, 16), 2, [2], 2),           # dblock4.0
    ("conv", 5, [64], 64, True, (4, 16, 16, 16), 2, [2], 2),           # dblock4.3, ublock1.4
    ("conv", 5, [64], 128, True, (4, 8, 8, 8), 2, [2], 2),             # cblock_center.0
    ("conv", 5, [128], 128, True, (4, 8, 8, 8), 2, [2], 2),            # cblock_center.3
    ("convt2", 2, [128], 128, True, (4, 8, 8, 8), 0, [0], 0),          # ublock1.0 (8^3: not fusable)
    ("conv", 5, [128], 64, True, (4, 16, 16, 16), 2, [2], 2),          # ublock1.1
    ("up", 5, [64, 64], 32, True, (4, 16, 16, 16), 1, [2, 2], 1),      # ublock2.0 + .1 (dgrad 256->64)
    ("up", 5, [32, 32], 16, True, (4, 32, 32, 32), 1, [1, 1], 1),      # ublock3.0 + .1 (dgrad 128->32)
    ("up", 5, [16, 16], 8, True, (4, 64, 64, 64), 1, [1, 1], 1),       # ublock4.0 + .1 (dgrad 64->16)
]

PROFILE_TABLES = ["profiles/r2_kernel_table_g_UNetSP.txt", "profiles/r2_kernel_table_e_recAE.txt"]


def _case_id(c):
    kind, k, chans, cout, _, (n, d, h, w) = c[:6]
    return "%s-k%d-%s-%d@%dx%dx%dx%d" % (kind, k, "+".join(map(str, chans)), cout, n, d, h, w)


def launch_labels(case):
    """The kernel-table labels of the launches one layer makes in a training step."""
    kind, k, chans, cout, _, (n, d, h, w) = case[:6]
    at = "@%dx%dx%dx%d" % (n, d, h, w)
    cin = sum(chans)
    if kind == "convt2":
        return {"ctu_convt2_%s %d->%d %s" % (p, cin, cout, at) for p in ("fprop", "dgrad", "wgrad")}
    if kind == "conv_fwd":
        return {"ctu_conv3d_fprop[tcgen05] k%d %d->%d %s" % (k, cin, cout, at)}
    if kind == "conv":
        out = {"ctu_conv3d_fprop[tcgen05] k%d %d->%d %s" % (k, cin, cout, at),
               "ctu_conv3d_wgrad[tcgen05] k%d %d->%d %s" % (k, cin, cout, at)}
        return out | {"ctu_conv3d_fprop[tcgen05] k%d %d->%d %s" % (k, cout, c, at) for c in chans}
    cop = (cout + 7) // 8 * 8
    out = {"ctu_conv3d_fprop[tcgen05][up-fused] k3 %d->%d %s" % (cin, cout, at),
           "ctu_conv3d_wgrad[tcgen05][up-fused] k3 %d->%d %s" % (cin, cop, at)}
    return out | {"ctu_conv3d_fprop[tcgen05] k3 %d->%d %s" % (8 * cop, c, at) for c in chans}


def test_layer_table_covers_the_profiled_launches():
    """Every ctu_conv3d_* / ctu_convt2_* row of the benchmarked step's kernel tables is a launch of a LAYERS case."""
    covered = set().union(*(launch_labels(c) for c in LAYERS))
    rows = []
    for name in PROFILE_TABLES:
        with open(os.path.join(ROOT, name)) as f:
            for line in f:
                m = re.match(r"(ctu_conv(?:3d|t2)_\S+ .*?@\S+)", line)
                if m:
                    rows.append(re.sub(r"\s+", " ", m.group(1)))
    assert len(rows) >= 60
    missing = [r for r in rows if r not in covered]
    assert not missing, missing


# ---------------------------------------------------------------------------------------------------------------------
def _check_stats(sums, y_stored, cout, phase_cout=None):
    """Fused BatchNorm sums (double [sum | sum of squares], 8-padded) against float64 sums of the stored outputs."""
    cpad = ((phase_cout or cout) + 7) // 8 * 8
    c = phase_cout or cout
    s, q = X.stats_ref(y_stored, phase_cout)
    yd = X.phase_to_natural(y_stored, phase_cout) if phase_cout else y_stored
    scale = yd.double().abs().sum((0, 2, 3, 4))
    got = sums.cpu()
    assert ((got[:c] - s).abs() <= 1e-6 * scale).all(), "BatchNorm sums: %s vs %s" % (got[:c], s)
    assert ((got[cpad:cpad + c] - q).abs() <= 1e-6 * q).all(), "BatchNorm sums of squares: %s vs %s" % (got[cpad:cpad + c], q)


def run_conv(family, k, chans, cout, bias, dims, tc_f=None, tc_d=None, tc_w=None, fwd_only=False, mode="bf16", seed=0):
    """One Conv3d through the Engine (the product's own dispatch) against the float32 CPU reference, bit for bit."""
    import ctunet_b200.engine as E
    n, d, h, w = dims
    g = torch.Generator().manual_seed(seed + 1000 * k + 10 * cout + sum(chans))
    xs = [X.operand(family, (n, c, d, h, w), g) for c in chans]
    cin = sum(chans)
    wt = X.operand(family, (cout, cin, k, k, k), g)
    bs = X.bias_operand(family, cout, g) if bias else None
    dy = X.operand(family, (n, cout, d, h, w), g)
    rnd = X.round_bf16 if mode == "bf16" else (lambda t: t)
    eng = E.Engine(torch.device(DEV), mode, record=not fwd_only)
    if tc_f is not None:
        assert eng.use_tc
        assert E.tc_variant(k, chans, cout, n, d, h, w) == tc_f
        assert [E.tc_variant(k, [cout], c, n, d, h, w) for c in chans][:len(tc_d)] == tc_d
        if not fwd_only:
            assert E.wgrad_variant(k, chans, cout, d, h, w) == tc_w
    acts = [eng.pack(x.to(DEV)) for x in xs]
    wg = wt.to(DEV).requires_grad_()
    bg = bs.to(DEV).requires_grad_() if bias else None
    y = eng.conv(acts, wg, bg, k, [True] * len(acts), bn_stats=True)
    yo = eng.unpack(y).cpu()
    xcat = torch.cat(xs, 1)
    X.exact_premise("fwd", x=xcat, w=wt, b=bs, k=k)
    yr = rnd(X.conv_fwd(xcat, wt, bs, k))
    X.assert_exact(yo, yr, "forward")
    _check_stats(y.sums, yr, cout)
    if fwd_only:
        return
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    dxs = [eng.unpack(eng.agrads[id(a)]).cpu() for a in acts]
    torch.cuda.synchronize()                 # weight gradients run on side streams
    dw = eng.pgrads[id(wg)].cpu()
    db = eng.pgrads[id(bg)].cpu() if bias else None
    X.exact_premise("dgrad", dy=dy, w=wt, k=k)
    for i, (got, r) in enumerate(zip(dxs, X.conv_dgrad(dy, wt, k, chans))):
        X.assert_exact(got, rnd(r), "dgrad of source %d" % i)
    if family == "T" or 9 * n * d * h * w < X.EXACT_LIMIT:
        X.exact_premise("wgrad", x=xcat, dy=dy, k=k)
        X.assert_exact(dw, X.conv_wgrad(xcat, dy, k), "wgrad")
        if bias:
            X.assert_exact(db, X.bias_grad(dy), "bias grad")


def run_convt2(family, cin, cout, dims, seed=0):
    """ConvTranspose3d(k2, s2) with bias (CUDA-core kernels) through the Engine against float64 autograd."""
    import torch.nn.functional as F
    from ctunet_b200.engine import Engine
    n, d, h, w = dims
    g = torch.Generator().manual_seed(seed + cin)
    x = X.operand(family, (n, cin, d, h, w), g)
    wt = X.operand(family, (cin, cout, 2, 2, 2), g)
    bs = X.bias_operand(family, cout, g)
    dy = X.operand(family, (n, cout, 2 * d, 2 * h, 2 * w), g)
    xr, wr, br = x.double().requires_grad_(), wt.double().requires_grad_(), bs.double().requires_grad_()
    yr = F.conv_transpose3d(xr, wr, br, 2)
    yr.backward(dy.double())
    assert yr.abs().max().item() < X.EXACT_LIMIT and xr.grad.abs().max().item() < X.EXACT_LIMIT
    eng = Engine(torch.device(DEV), "bf16", record=True)
    a = eng.pack(x.to(DEV))
    wg, bg = wt.to(DEV).requires_grad_(), bs.to(DEV).requires_grad_()
    y = eng.convt([a], wg, bg, [True])
    X.assert_exact(eng.unpack(y).cpu(), X.round_bf16(yr.detach().float()), "convT forward")
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    X.assert_exact(eng.unpack(eng.agrads[id(a)]).cpu(), X.round_bf16(xr.grad.float()), "convT dgrad")
    torch.cuda.synchronize()
    if family == "T" or 9 * 8 * n * d * h * w < X.EXACT_LIMIT:
        X.assert_exact(eng.pgrads[id(wg)].cpu(), wr.grad.float(), "convT wgrad")
        X.assert_exact(eng.pgrads[id(bg)].cpu(), br.grad.float(), "convT bias grad")


def _close_or_exact(got, exp64, bound, what):
    """Bit-exact where the integer premise holds (every |partial sum| below 2^24), else within 1e-6 per element relative to
    ``bound``, the same sum over absolute values (fp32 rounding of a sum is relative to its terms, not to its result)."""
    if bound.max().item() < X.EXACT_LIMIT:
        X.assert_exact(got, exp64.float(), what)
    else:
        err = (got.double() - exp64).abs()
        assert (err <= 1e-6 * bound).all(), "%s: max err %.3e" % (what, err.max().item())


def run_up(family, k, chans, cout, bias3, dims, tc_f=None, tc_d=None, tc_w=None, seed=0):
    """The fused up-sampling stage through Engine.up_conv: phase-major output against the composed reference (pad rows
    exactly 0), BatchNorm sums over phases, data gradients, and the decomposed weight gradients dWT, dbT, dW3 (, db3)."""
    import ctunet_b200.engine as E
    from ctunet_b200 import _lib
    n, d, h, w = dims
    lib = _lib.load()
    g = torch.Generator().manual_seed(seed + 77 * k + cout)
    cin = sum(chans)
    co8 = lib.ctu_upfuse_cout(cout)
    # P: non-negative activations and gradients, ternary weights (the composed weights of {0..3} operands break the premise)
    xs = [X.operand(family, (n, c, d, h, w), g) for c in chans]
    dy_nat = X.operand(family, (n, cout, 2 * d, 2 * h, 2 * w), g)
    ct = nn.ConvTranspose3d(cin, cin, 2, 2)
    cv = nn.Conv3d(cin, cout, k, 1, k // 2, bias=bias3)
    with torch.no_grad():
        ct.weight.copy_(X.ternary(ct.weight.shape, g))
        ct.bias.copy_(X.ternary_bias(cin, g))
        cv.weight.copy_(X.ternary(cv.weight.shape, g))
        if bias3:
            cv.bias.copy_(X.ternary_bias(cout, g))
    wt, bt, w3 = ct.weight.detach().clone(), ct.bias.detach().clone(), cv.weight.detach().clone()
    b3 = cv.bias.detach().clone() if bias3 else None
    chans1 = chans + [1]
    if tc_f is not None:
        assert E.tc_variant(3, chans1, co8, n, d, h, w) == tc_f
        assert [E.tc_variant(3, [co8], c, n, d, h, w) for c in chans] == tc_d
        assert E.wgrad_variant(3, chans1, co8, d, h, w, cout if k == 3 else 0) == tc_w
    eng = E.Engine(torch.device(DEV), "bf16", record=True)
    ctg, cvg = ct.to(DEV), cv.to(DEV)
    acts = [eng.pack(x.to(DEV)) for x in xs]
    assert eng.up_fusable(acts, cout, k)
    y = eng.up_conv(acts, ctg, cvg, k, [True] * len(acts), True)
    assert y.c == co8 and y.c_nat == cout
    yo = eng.unpack(y).cpu()
    # reference: cat(srcs, ones) through the composed weights (float64 composition, rounded to bf16)
    wn = X.composed_weights(wt, bt, w3, k)
    b3n = X.composed_bias(b3, cout) if bias3 else None
    xo = X.with_ones(xs)
    X.exact_premise("fwd", x=xo, w=wn, b=b3n, k=3)
    yr = X.round_bf16(X.conv_fwd(xo, wn, b3n, 3))
    X.assert_exact(yo, yr, "fused forward (phase-major; pad rows 0)")
    _check_stats(y.sums, yr, co8, phase_cout=cout)
    dy = X.natural_to_phase(dy_nat, cout)
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    dxs = [eng.unpack(eng.agrads[id(a)]).cpu() for a in acts]
    torch.cuda.synchronize()
    X.exact_premise("dgrad", dy=dy, w=wn, k=3)
    for i, (got, r) in enumerate(zip(dxs, X.conv_dgrad(dy, wn, 3, chans1))):
        X.assert_exact(got, X.round_bf16(r), "fused dgrad of source %d" % i)
    if not (family == "T" or 9 * n * d * h * w < X.EXACT_LIMIT):
        return
    X.exact_premise("wgrad", x=xo, dy=dy, k=3)
    dwn = X.conv_wgrad(xo, dy, 3).double()
    dbn = X.bias_grad(dy).double()
    # the decomposition is the chain rule of the composition: its exact value and a bound from absolute values
    wt64, bt64, w364 = (t.double().requires_grad_() for t in (wt, bt, w3))
    grads = torch.autograd.grad(X.U.compose(wt64, bt64, w364, k), [wt64, bt64, w364], dwn.view(co8, cin + 1, 3, 3, 3))
    awt, abt, aw3 = (t.double().abs().requires_grad_() for t in (wt, bt, w3))
    bounds = torch.autograd.grad(X.U.compose(awt, abt, aw3, k), [awt, abt, aw3], dwn.abs().view(co8, cin + 1, 3, 3, 3))
    for prm, exp, bnd, what in ((ctg.weight, grads[0], bounds[0], "dWT"), (ctg.bias, grads[1], bounds[1], "dbT"),
                                (cvg.weight, grads[2], bounds[2], "dW3")):
        _close_or_exact(eng.pgrads[id(prm)].cpu(), exp, bnd, what)
    if bias3:
        X.assert_exact(eng.pgrads[id(cvg.bias)].cpu(), dbn.view(8, -1)[:, :cout].sum(0).float(), "db3")


def run_case(family, case):
    kind, k, chans, cout, bias, dims, tc_f, tc_d, tc_w = case
    if kind == "convt2":
        run_convt2(family, chans[0], cout, dims)
    elif kind == "up":
        run_up(family, k, list(chans), cout, bias, dims, tc_f, tc_d, tc_w)
    else:
        run_conv(family, k, list(chans), cout, bias, dims, tc_f, tc_d, tc_w, fwd_only=(kind == "conv_fwd"))


@gpu
@pytest.mark.parametrize("family", ["T", "P"])
@pytest.mark.parametrize("case", LAYERS, ids=_case_id)
def test_benchmarked_layer_is_bit_exact(case, family):
    run_case(family, case)


# ---------------------------------------------------------------------------------------------------------------------
# (b) Fused stages at kernel level: the phase-sparse weight gradient, and the composed forward against the unfused
# ConvTranspose3d -> Conv3d where the composed weights are exact in bf16.
UP_KERNEL_CASES = [
    (3, [14, 14], 7, (1, 5, 16, 16)),
    (3, [28, 28], 14, (3, 3, 16, 32)),      # phase-sparse with 2 output blocks per phase
    (3, [56, 56], 28, (1, 3, 16, 16)),      # 4 blocks per phase: groups of one (qd, qh)
    (3, [6], 5, (3, 17, 16, 16)),           # one source, ragged d-chunks
]


@gpu
@pytest.mark.parametrize("family", ["T", "P"])
@pytest.mark.parametrize("case", UP_KERNEL_CASES, ids=lambda c: "%d-%s-%d" % (c[0], "+".join(map(str, c[1])), c[2]))
def test_fused_stage_kernels_bit_exact(case, family):
    import torch.nn.functional as F
    from ctunet_b200 import _lib
    from ctunet_b200._lib import call, int_array, ptr_array, stream_ptr
    from ctunet_b200.engine import Engine
    k, chans, cout, (n, d, h, w) = case
    lib = _lib.load()
    g = torch.Generator().manual_seed(5 * cout + n)
    cin = sum(chans)
    co8 = lib.ctu_upfuse_cout(cout)
    chans1 = chans + [1]
    xs = [X.operand(family, (n, c, d, h, w), g) for c in chans]
    density = min(0.5, 16.0 / cin)          # sparse enough that most draws keep the composed weights within 256
    wt, bt = X.ternary((cin, cin, 2, 2, 2), g, density), X.ternary_bias(cin, g)
    w3 = X.ternary((cout, cin, k, k, k), g, density)
    wn = X.composed_weights(wt, bt, w3, k)
    xo = X.with_ones(xs)
    eng = Engine(torch.device(DEV), "bf16", record=False)
    acts = [eng.pack(x.to(DEV)) for x in xs] + [eng.pack(torch.ones(n, 1, d, h, w, device=DEV))]
    wk = eng._kernel_weights_chain(wn.to(DEV), co8, 3, chans1, 1)
    y = eng.new_act(co8, n, d, h, w)
    y.buf.fill_(0.5)                         # not a possible result: every element must be written
    call("ctu_conv3d_fprop", eng.dtype, ptr_array([a.ptr for a in acts]), int_array(chans1), len(acts), wk.data_ptr(), None,
         y.ptr, None, 0, co8, 3, n, d, h, w, 1, stream_ptr())
    yo = eng.unpack(y).cpu()
    X.exact_premise("fwd", x=xo, w=wn, k=3)
    yr = X.round_bf16(X.conv_fwd(xo, wn, None, 3))
    cop = co8 // 8
    assert torch.equal(yo.view(n, 8, cop, d, h, w)[:, :, cout:], torch.zeros(n, 8, cop - cout, d, h, w)), "pad rows"
    X.assert_exact(yo, yr, "composed forward")
    if wn.abs().max().item() <= 256:         # the bf16 composed weights are the exact ones: the fusion is exact end to end
        ref = F.conv3d(F.conv_transpose3d(torch.cat(xs, 1).double(), wt.double(), bt.double(), 2), w3.double(), None, 1, 1)
        X.assert_exact(X.phase_to_natural(yo, cout), X.round_bf16(ref.float()), "unfused ConvTranspose3d -> Conv3d")
    # phase-sparse weight gradient: bit for bit on the structural support (the other entries are unspecified)
    dy = X.natural_to_phase(X.operand(family, (n, cout, 2 * d, 2 * h, 2 * w), g), cout)
    dya = eng.pack(dy.to(DEV))
    ca = int_array(chans1)
    dwp = torch.empty(lib.ctu_conv_wpack_floats(co8, 3, len(chans1), ca), device=DEV)
    dbn = torch.empty(co8, device=DEV)
    dwn = torch.empty(co8, cin + 1, 3, 3, 3, device=DEV)
    call("ctu_conv3d_wgrad", eng.dtype, ptr_array([a.ptr for a in acts]), ca, len(acts), dya.ptr, dwp.data_ptr(),
         dbn.data_ptr(), cout, co8, 3, n, d, h, w, 1, stream_ptr())
    call("ctu_conv_unpack_wgrad", dwp.data_ptr(), dwn.data_ptr(), co8, 3, len(chans1), ca, stream_ptr())
    X.exact_premise("wgrad", x=xo, dy=dy, k=3)
    sup = X.structural_support(cin, cout)
    X.assert_exact(dwn.cpu()[sup], X.conv_wgrad(xo, dy, 3)[sup], "phase-sparse wgrad on the support")
    X.assert_exact(dbn.cpu(), X.bias_grad(dy), "phase-major bias grad")


# ---------------------------------------------------------------------------------------------------------------------
# (c) Edge geometries, batch 1 and 3 (k, source channels, cout, bias, (d, h, w)).
EDGE_CASES = [
    (3, [7], 7, False, (1, 16, 32)),        # d = 1: one plane, every tap but the centre plane reads padding
    (3, [7], 7, True, (2, 16, 16)),         # d = 2 (tap-stationary weight gradient at 16 x 16)
    (3, [14], 14, False, (17, 32, 32)),     # d prime: ragged d-chunks and plane shares
    (5, [8], 8, True, (17, 16, 32)),        # ... 5^3, two-CTA one-block kernel
    (3, [7], 14, False, (4, 16, 48)),       # h != w: 1 x 3 tiles per plane
    (3, [14], 7, False, (4, 32, 16)),       # 2 x 1 tiles
    (3, [2], 13, True, (3, 16, 16)),        # pad lanes in input (2 of 8) and output (13 of 16) blocks
    (3, [13], 2, False, (3, 16, 16)),
    (3, [28], 7, False, (3, 16, 32)),       # 28 channels: 4 blocks, the last half padding
    (3, [24], 24, False, (3, 16, 32)),      # odd number of input blocks (3): the tap-paired tail
    (3, [56], 14, False, (3, 16, 32)),      # 7 input blocks: staged in groups of four, short last group (4 + 3)
    (3, [24, 40], 8, False, (3, 16, 16)),   # 8 blocks over two sources, groups of four; output cobg 1
    (3, [14], 16, False, (3, 16, 32)),      # output cobg 2
    (3, [14], 40, False, (3, 16, 32)),      # output cobg 4 with a partial second group (5 blocks)
    (5, [8], 16, True, (3, 16, 32)),        # 5^3 output cobg 2
    (5, [8], 24, True, (3, 16, 32)),        # 5^3 cobg 2 with a partial second group
    (3, [40], 16, False, (3, 32, 32)),      # wgrad: 5 input blocks balanced as 3 + 2
    (5, [56], 56, True, (3, 32, 32)),       # wgrad: output-channel groups 16, 16, 16, 8
    (3, [7], 7, False, (3, 8, 8)),          # 8 x 8 planes: weight-streaming forward, tap-stationary wgrad
    (3, [56], 56, False, (3, 16, 16)),      # weight-streaming at 16 x 16 (preferred for wide layers)
    (5, [16], 24, True, (3, 8, 8)),
    (3, [40], 48, False, (3, 32, 32)),      # resident-weights kernel above 16 x 16 with many channels
]


@gpu
@pytest.mark.parametrize("family", ["T", "P"])
@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("case", EDGE_CASES, ids=lambda c: "k%d-%s-%d-%dx%dx%d" % ((c[0], "+".join(map(str, c[1])), c[2]) + c[4]))
def test_edge_geometry_is_bit_exact(case, n, family):
    from ctunet_b200.engine import tc_variant
    k, chans, cout, bias, (d, h, w) = case
    assert tc_variant(k, chans, cout, n, d, h, w) > 0           # a tensor kernel, not the CUDA-core fallback
    run_conv(family, k, chans, cout, bias, (n, d, h, w), seed=n)


@gpu
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("case", [(3, [7, 5], 9, True, (3, 5, 8, 12)), (5, [4], 6, True, (1, 6, 12, 8)),
                                  (3, [2], 7, False, (3, 17, 16, 16))])
def test_direct_path_is_bit_exact(case, mode):
    """The CUDA-core kernels (CONV_PATH = "direct"): the integer premise holds in fp32 check mode too."""
    import ctunet_b200.engine as E
    k, chans, cout, bias, dims = case
    old = E.CONV_PATH
    E.CONV_PATH = "direct"
    try:
        for family in ("T", "P"):
            run_conv(family, k, chans, cout, bias, dims, mode=mode)
    finally:
        E.CONV_PATH = old


# ---------------------------------------------------------------------------------------------------------------------
# (d) Every output element written, pad lanes zero (the layout invariant of include/ctunet_b200.h).
@gpu
@pytest.mark.parametrize("tc,case", [(1, (3, 7, 13, (2, 5, 16, 32))), (1, (5, 8, 13, (1, 17, 16, 16))),
                                     (1, (3, 56, 21, (3, 3, 32, 16))), (2, (3, 56, 13, (2, 4, 16, 16))),
                                     (2, (5, 64, 61, (3, 5, 8, 8)))])
def test_fprop_writes_every_output_element(tc, case):
    from ctunet_b200._lib import call, int_array, ptr_array, stream_ptr
    from ctunet_b200.engine import Engine, tc_variant
    k, cin, cout, (n, d, h, w) = case
    assert tc_variant(k, [cin], cout, n, d, h, w) == tc or tc == 1
    g = torch.Generator().manual_seed(cin * cout)
    x = X.ternary((n, cin, d, h, w), g)
    wt = X.ternary((cout, cin, k, k, k), g)
    eng = Engine(torch.device(DEV), "bf16", record=False)
    xa = eng.pack(x.to(DEV))
    wk = eng._kernel_weights_chain(wt.to(DEV), cout, k, [cin], tc, dims=(n, d, h, w))
    y = eng.new_act(cout, n, d, h, w)
    y.buf.fill_(0.5)                         # with integer operands 0.5 cannot be a result
    call("ctu_conv3d_fprop", eng.dtype, ptr_array([xa.ptr]), int_array([cin]), 1, wk.data_ptr(), None, y.ptr, None, 0,
         cout, k, n, d, h, w, tc, stream_ptr())
    torch.cuda.synchronize()
    buf = y.buf.float().cpu()
    assert not (buf == 0.5).any(), "%d elements not written" % int((buf == 0.5).sum())
    assert torch.equal(buf[:, -1, ..., cout % 8:], torch.zeros_like(buf[:, -1, ..., cout % 8:])), "pad lanes"
    X.assert_exact(eng.unpack(y).cpu(), X.round_bf16(X.conv_fwd(x, wt, None, k)), "forward")
