"""The oracle of the bit-exact convolution tests (conv_exact_oracle.py) checked on the CPU: the float32 references equal
float64 on integer operands, bf16 rounding is round-to-nearest-even, the composed low-resolution convolution equals
ConvTranspose3d -> Conv3d, and the structural support of the composed weights is what the tap algebra says."""
import itertools

import pytest
import torch
import torch.nn.functional as F

import conv_exact_oracle as X


@pytest.mark.parametrize("family", ["T", "P"])
@pytest.mark.parametrize("k,chans,cout,bias", [(3, [7], 5, False), (3, [6, 3], 9, True), (5, [4], 3, True),
                                               (5, [2, 5, 1], 6, False)])
def test_float32_reference_equals_float64(family, k, chans, cout, bias):
    """Under the premise every fp32 partial sum is an exact integer: forward, data, weight and bias gradients of the
    float32 references equal float64 autograd bit for bit."""
    g = torch.Generator().manual_seed(k * 100 + cout)
    n, d, h, w = 2, 5, 8, 12
    xs = [X.operand(family, (n, c, d, h, w), g) for c in chans]
    cin = sum(chans)
    wt = X.operand(family, (cout, cin, k, k, k), g)
    b = X.bias_operand(family, cout, g) if bias else None
    dy = X.operand(family, (n, cout, d, h, w), g)
    X.exact_premise("fwd", x=torch.cat(xs, 1), w=wt, b=b, k=k)
    X.exact_premise("dgrad", dy=dy, w=wt, k=k)
    X.exact_premise("wgrad", x=torch.cat(xs, 1), dy=dy, k=k)
    xd = [x.double().requires_grad_() for x in xs]
    wd = wt.double().requires_grad_()
    bd = b.double().requires_grad_() if bias else None
    yd = F.conv3d(torch.cat(xd, 1), wd, bd, 1, k // 2)
    yd.backward(dy.double())
    X.assert_exact(X.conv_fwd(xs, wt, b, k), yd.detach().float(), "forward")
    for got, r in zip(X.conv_dgrad(dy, wt, k, chans), xd):
        X.assert_exact(got, r.grad.float(), "dgrad")
    X.assert_exact(X.conv_wgrad(torch.cat(xs, 1), dy, k), wd.grad.float(), "wgrad")
    if bias:
        X.assert_exact(X.bias_grad(dy), bd.grad.float(), "bias grad")


def test_round_bf16_ties_to_even():
    t = torch.tensor([257.0, 259.0, 770.0, 774.0, 256.0, 258.0, -257.0, -259.0])
    assert X.round_bf16(t).tolist() == [256.0, 260.0, 768.0, 776.0, 256.0, 258.0, -256.0, -260.0]


def test_premise_rejects_sums_beyond_2_24():
    x = torch.ones(1, 64, 8, 16, 16)
    w = torch.full((1, 64, 5, 5, 5), 2.0 ** 12)
    with pytest.raises(AssertionError, match="premise"):
        X.exact_premise("fwd", x=x, w=w, k=5)
    assert X.exact_premise("fwd", x=x, w=torch.ones(1, 64, 5, 5, 5), k=5) == 64 * 125


@pytest.mark.parametrize("k,chans,cout,bias3", [(3, [6], 5, False), (3, [4, 4], 9, True), (5, [3, 3], 4, True)])
def test_composed_convolution_equals_convT_then_conv(k, chans, cout, bias3):
    """Integer weights whose composed magnitude is at most 256 are exact in bf16: cat(srcs, ones) through the composed
    low-resolution convolution, mapped back from phase-major channels, equals conv_transpose3d -> conv3d bit for bit."""
    g = torch.Generator().manual_seed(7 * k + cout)
    n, d, h, w = 2, 3, 4, 5
    cin = sum(chans)
    xs = [X.ternary((n, c, d, h, w), g) for c in chans]
    wt = X.ternary((cin, cin, 2, 2, 2), g)
    bt = X.ternary_bias(cin, g)
    w3 = X.ternary((cout, cin, k, k, k), g)
    b3 = X.ternary_bias(cout, g) if bias3 else None
    wn = X.composed_weights(wt, bt, w3, k)
    assert wn.abs().max().item() <= 256
    exact = torch.equal(wn.double(), X.U.compose(wt.double(), bt.double(), w3.double(), k))
    assert exact
    xo = X.with_ones(xs)
    X.exact_premise("fwd", x=xo, w=wn, b=X.composed_bias(b3, cout) if bias3 else None, k=3)
    y = X.conv_fwd(xo, wn, X.composed_bias(b3, cout) if bias3 else None, 3)
    cop = (cout + 7) // 8 * 8
    assert torch.equal(y.view(n, 8, cop, d, h, w)[:, :, cout:], torch.zeros(n, 8, cop - cout, d, h, w))   # pad rows
    ref = F.conv3d(F.conv_transpose3d(torch.cat(xs, 1).double(), wt.double(), bt.double(), 2), w3.double(),
                   b3.double() if bias3 else None, 1, k // 2)
    X.assert_exact(X.phase_to_natural(y, cout), ref.float(), "fused stage")
    X.assert_exact(X.natural_to_phase(ref.float(), cout), y, "phase mapping")


@pytest.mark.parametrize("cin,cout", [(3, 5), (8, 8), (2, 13)])
def test_structural_support_matches_tap_enumeration(cin, cout):
    """Per dimension, output phase q of a 3-tap convolution after a stride-2 transposed one reads low-resolution offsets
    floor((q + kk - 1) / 2), kk = 0..2: {-1, 0} for q = 0 and {0, 1} for q = 1.  Pad rows (co >= cout) have no support."""
    cop = (cout + 7) // 8 * 8
    exp = torch.zeros(8, cop, cin + 1, 3, 3, 3, dtype=torch.bool)
    for qd, qh, qw in itertools.product(range(2), repeat=3):
        for kd, kh, kw in itertools.product(range(3), repeat=3):
            dd, dh, dw = ((q + kk - 1) // 2 for q, kk in ((qd, kd), (qh, kh), (qw, kw)))
            exp[qd * 4 + qh * 2 + qw, :cout, :, dd + 1, dh + 1, dw + 1] = True
    sup = X.structural_support(cin, cout)
    assert torch.equal(sup, exp.view(8 * cop, cin + 1, 3, 3, 3))
    assert int(sup.sum()) == 8 * cout * (cin + 1) * 8          # 2 of 3 offsets per dimension


def test_mismatch_report_names_voxel_tile_and_plane():
    exp = torch.zeros(2, 3, 4, 32, 48)
    got = exp.clone()
    got[1, 2, 3, 17, 40] = 1.0
    count, where = X.mismatches(got, exp)
    assert count == 1
    assert where[0].startswith("(n=1, c=2, z=3, y=17, x=40) tile (1, 2) plane 3")
    with pytest.raises(AssertionError, match="1 of 36864 elements differ"):
        X.assert_exact(got, exp, "planted")
