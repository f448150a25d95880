"""tcgen05/TMA implicit-GEMM convolution (conv_tc.cu) against fp32 PyTorch on the CPU and against the
CUDA-core direct kernel, on the layer shapes of the networks (GPU)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"

# (k, cin, cout, bias, (n, d, h, w))
CASES = [
    (3, 2, 7, False, (1, 4, 16, 16)),
    (3, 7, 7, False, (2, 9, 32, 16)),
    (3, 14, 14, False, (1, 8, 16, 32)),
    (3, 28, 7, False, (1, 6, 16, 16)),
    (3, 7, 14, False, (1, 3, 16, 16)),
    (3, 14, 28, False, (1, 5, 32, 32)),
    (3, 56, 14, False, (1, 4, 16, 16)),      # odd number of channel blocks (7): tap-paired tail
    (3, 24, 24, False, (1, 4, 16, 16)),      # 3 blocks
    (3, 28, 28, False, (1, 40, 16, 16)),     # several d-chunks
    (5, 1, 8, True, (1, 6, 16, 16)),
    (5, 8, 8, True, (1, 5, 16, 32)),
    (5, 16, 8, True, (1, 4, 16, 16)),
    (3, 7, 7, True, (1, 2, 16, 16)),
    (3, 7, 7, False, (1, 1, 16, 16)),
    (3, 56, 56, False, (1, 3, 16, 16)),      # wgrad: several input-block groups
    (3, 112, 28, False, (1, 2, 16, 16)),
    (3, 28, 112, False, (1, 2, 16, 16)),     # wgrad: output channels split over TMEM
    (5, 14, 28, True, (1, 3, 16, 16)),
    (5, 56, 56, True, (1, 3, 16, 16)),       # wgrad: partial last output-channel group (16,16,16,8); fprop: wide kernel
    # the benchmarked grids (batch 4 x 128^3 runs these shapes per sample): d = 128 (balanced plane shares, TcWalk; fixed d-chunks below 16 planes per CTA), 8 x 8 tiles of
    # 16 x 16 per plane, persistent 296-CTA schedules
    (3, 2, 7, False, (1, 128, 128, 128)),
    (3, 7, 7, False, (2, 128, 128, 128)),
    (3, 14, 14, False, (2, 64, 64, 64)),
    (3, 7, 14, False, (1, 64, 64, 64)),
    (5, 8, 8, True, (1, 48, 128, 128)),
    (5, 1, 8, True, (1, 128, 128, 128)),
]

# wide, low-resolution layers: the weight-streaming kernel (conv_wide.cu), M = 128 tiles at 16^3, M = 64 at 8^3
WIDE_CASES = [
    (5, 64, 64, True, (2, 4, 16, 16)),
    (5, 128, 64, True, (1, 3, 16, 16)),      # two channel groups of 8 blocks
    (5, 112, 56, True, (1, 4, 16, 16)),      # groups of 8 + 6 blocks, 7 output blocks
    (5, 64, 128, True, (2, 8, 8, 8)),        # 8 x 8 planes: M = 64
    (5, 128, 128, True, (1, 8, 8, 8)),
    (5, 56, 112, True, (1, 5, 8, 8)),        # odd block count: dummy K chunk
    (3, 56, 112, False, (2, 8, 8, 8)),       # generic UNet center block (dead branch)
    (3, 112, 112, False, (1, 8, 8, 8)),
    (3, 56, 56, False, (4, 16, 16, 16)),     # both kernels cover it: the wide one is preferred
    (3, 7, 7, False, (1, 2, 8, 8)),          # below the preference threshold, but the only tensor kernel for 8 x 8
    (3, 40, 48, False, (1, 3, 32, 32)),      # the resident-weights kernel (preferred above 16 x 16)
]


def _bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _conv64(x, w, b, k):
    """float64 conv3d(x, w) + b and its magnitude |w| (*) |x| + |b|, in d-slabs of at most 16 planes (plus the halo) so
    that the float64 column buffers of the 128^3 cases stay small."""
    p = k // 2
    n, c, d, h, wd = x.shape
    x, w = x.double(), w.double()
    b = b.double() if b is not None else None
    slab = max(1, min(16, (1 << 26) // (c * k ** 3 * h * wd)))
    ys, bs = [], []
    for z0 in range(0, d, slab):
        z1 = min(d, z0 + slab)
        lo, hi = max(0, z0 - p), min(d, z1 + p)
        xs = F.pad(x[:, :, lo:hi], (0, 0, 0, 0, lo - (z0 - p), (z1 + p) - hi))
        ys.append(F.conv3d(xs, w, b, 1, (0, p, p)))
        bs.append(F.conv3d(xs.abs(), w.abs(), b.abs() if b is not None else None, 1, (0, p, p)))
    return torch.cat(ys, 2), torch.cat(bs, 2)


def _check_elementwise(got, x, w, b, k, what):
    """|y - y64| <= 2^-8 |y64| + 2^-16 (|w| (*) |x| + |b|) per element, y64 the float64 result on the bf16-rounded operands:
    one bf16 rounding of the output (at most 2^-8 relative) plus fp32 accumulation error.  Returns the worst ratio to the
    bound (printed, so that the rounding model can be compared with what the B200 does)."""
    ref, mag = _conv64(x, w, b, k)
    err = (got.double() - ref).abs()
    bound = 2.0 ** -8 * ref.abs() + 2.0 ** -16 * mag
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), err * float("inf")).nan_to_num(0.0)
    worst = ratio.max().item()
    print("%s: worst |err| / bound %.3f" % (what, worst))
    if worst > 1.0:
        idx = tuple(int(i) for i in (ratio == ratio.max()).nonzero()[0])
        raise AssertionError("%s: |err| %.3e > bound %.3e at %s (ratio %.3f)" % (what, err[idx].item(), bound[idx].item(),
                                                                                 idx, worst))
    return worst


def _dgrad_weights(w):
    """The data gradient is a convolution of dy with the flipped, transposed weights."""
    return w.flip(2, 3, 4).transpose(0, 1)


@pytest.mark.parametrize("case", CASES + WIDE_CASES)
def test_tc_conv_matches_reference(case):
    from ctunet_b200.engine import Engine, tc_variant
    from ctunet_b200 import _lib
    k, cin, cout, use_bias, (n, d, h, w) = case
    assert _lib.load().ctu_has_tensor_path() == 1
    fprop_on_tc = tc_variant(k, [cin], cout, n, d, h, w)
    from ctunet_b200.engine import WIDE_MAX_HW, WIDE_MIN_CH, tc_supported
    wide = (not tc_supported(k, [cin], cout, d, h, w)) or (min(cin, cout) >= WIDE_MIN_CH and max(h, w) <= WIDE_MAX_HW)
    assert fprop_on_tc == (2 if wide else 1)
    assert wide or case not in WIDE_CASES[:-2]
    assert tc_variant(k, [cout], cin, n, d, h, w) > 0        # the data gradient runs on the tensor cores too
    g = torch.Generator().manual_seed(k * 100 + cin)
    x = _bf(torch.randn(n, cin, d, h, w, generator=g))
    wt = torch.randn(cout, cin, k, k, k, generator=g) / (cin * k ** 3) ** 0.5
    bs = torch.randn(cout, generator=g) if use_bias else None
    dy = _bf(torch.randn(n, cout, d, h, w, generator=g))

    eng = Engine(torch.device(DEV), "bf16", record=True)
    assert eng.use_tc
    wg = wt.to(DEV).requires_grad_()
    bg = bs.to(DEV).requires_grad_() if use_bias else None
    xa = eng.pack(x.to(DEV))
    y = eng.conv([xa], wg, bg, k, [True], bn_stats=True)
    yo = eng.unpack(y).cpu()
    scale = yo.abs().max().item()
    _check_elementwise(yo, x, _bf(wt), bs, k, "fprop %s" % (case,))     # the tensor path rounds the weights to bf16
    # fused BatchNorm statistics = sums of the stored (bf16-rounded) outputs
    sums = y.sums.cpu()
    cpad = (cout + 7) // 8 * 8
    ref_sum = yo.double().sum((0, 2, 3, 4))
    ref_sq = (yo.double() ** 2).sum((0, 2, 3, 4))
    assert torch.allclose(sums[:cout], ref_sum, rtol=1e-4, atol=1e-2 * scale)
    assert torch.allclose(sums[cpad:cpad + cout], ref_sq, rtol=1e-4, atol=1e-3)
    # data gradient through the same kernel (flipped / transposed weights)
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    dx = eng.unpack(eng.agrads[id(xa)]).cpu()
    _check_elementwise(dx, dy, _dgrad_weights(_bf(wt)), None, k, "dgrad %s" % (case,))
    # weight gradient on the tensor cores (voxels as the K dimension): bf16 products, fp32 accumulation
    assert _lib.load().ctu_conv_tc_wgrad_supported(k, 1, _lib.int_array([cin]), cout, d, h, w) == (1 if h % 16 == 0 else 0)
    assert h % 16 == 0 or _lib.load().ctu_conv_wide_wgrad_supported(k, cin, cout, d, h, w) == 1   # 8 x 8: tap-stationary kernel
    wr = wt.clone().requires_grad_()
    br = bs.clone().requires_grad_() if use_bias else None
    F.conv3d(x, wr, br, 1, k // 2).backward(dy)
    dw = eng.pgrads[id(wg)].cpu()
    ws = wr.grad.abs().max().item()
    werr = (dw - wr.grad).abs().max().item()
    assert werr <= 2e-3 * ws, "wgrad err %.3e (scale %.3e)" % (werr, ws)
    if use_bias:
        db = eng.pgrads[id(bg)].cpu()
        assert (db - br.grad).abs().max().item() <= 2e-3 * br.grad.abs().max().item()


@pytest.mark.parametrize("case", [(3, 56, 56, (4, 16, 16, 16)), (5, 64, 64, (2, 16, 16, 16)), (5, 128, 64, (1, 6, 16, 16)),
                                  (3, 28, 56, (2, 16, 16, 16)), (5, 56, 112, (3, 8, 8, 8)), (3, 24, 40, (1, 5, 16, 24))])
def test_tap_stationary_wgrad_matches_reference(case):
    """conv3d_wgrad_small_kernel (use_tensor_path = 2) called directly: 8x8 tiles of 16-wide planes, d-planes split over CTAs."""
    from ctunet_b200 import _lib
    from ctunet_b200._lib import call, int_array, ptr_array, stream_ptr
    from ctunet_b200.engine import Engine
    k, cin, cout, (n, d, h, w) = case
    lib = _lib.load()
    assert lib.ctu_conv_wide_wgrad_supported(k, cin, cout, d, h, w) == 1
    g = torch.Generator().manual_seed(cin + cout)
    x = _bf(torch.randn(n, cin, d, h, w, generator=g))
    dy = _bf(torch.randn(n, cout, d, h, w, generator=g))
    wr = torch.zeros(cout, cin, k, k, k, requires_grad=True)
    br = torch.zeros(cout, requires_grad=True)
    F.conv3d(x, wr, br, 1, k // 2).backward(dy)
    eng = Engine(torch.device(DEV), "bf16", record=False)
    xa, dya = eng.pack(x.to(DEV)), eng.pack(dy.to(DEV))
    ca = int_array([cin])
    dwp = torch.empty(lib.ctu_conv_wpack_floats(cout, k, 1, ca), device=DEV)
    db = torch.empty(cout, device=DEV)
    dw = torch.empty(cout, cin, k, k, k, device=DEV)
    call("ctu_conv3d_wgrad", 1, ptr_array([xa.ptr]), ca, 1, dya.ptr, dwp.data_ptr(), db.data_ptr(), 0, cout, k, n, d, h, w, 2,
         stream_ptr())
    call("ctu_conv_unpack_wgrad", dwp.data_ptr(), dw.data_ptr(), cout, k, 1, ca, stream_ptr())
    assert (dw.cpu() - wr.grad).abs().max().item() <= 2e-3 * wr.grad.abs().max().item()
    assert (db.cpu() - br.grad).abs().max().item() <= 2e-3 * br.grad.abs().max().item()


def test_tc_and_direct_agree_on_network_layer():
    """Same bf16 inputs through both kernels: only weight rounding and accumulation order differ."""
    import ctunet_b200.engine as E
    g = torch.Generator().manual_seed(3)
    x = _bf(torch.rand(2, 7, 8, 32, 32, generator=g))
    wt = (torch.randn(7, 7, 3, 3, 3, generator=g) * 0.1).to(DEV)
    outs = []
    for path in ("auto", "direct"):
        E.CONV_PATH = path
        try:
            eng = E.Engine(torch.device(DEV), "bf16", record=False)
            outs.append(eng.unpack(eng.conv([eng.pack(x.to(DEV))], wt, None, 3, [False])).cpu())
        finally:
            E.CONV_PATH = "auto"
    assert (outs[0] - outs[1]).abs().max().item() <= 1e-2 * outs[1].abs().max().item()


def test_unsupported_shapes_fall_back_to_direct():
    from ctunet_b200.engine import tc_supported
    assert not tc_supported(3, [7], 7, 8, 8, 8)          # h, w not multiples of 16
    from ctunet_b200.engine import tc_variant
    assert tc_variant(3, [7], 7, 1, 8, 8, 8) == 2        # ... the weight-streaming kernel takes 8 x 8 planes
    assert tc_variant(3, [7], 7, 1, 12, 12, 12) == 0
    assert not tc_supported(1, [7], 7, 16, 16, 16)       # 1x1x1 is the head kernel's job
    assert tc_supported(3, [7, 7], 7, 16, 16, 16)        # concatenated sources: one tensor map per source
    assert not tc_supported(3, [7] * 5, 7, 16, 16, 16)   # at most CTU_MAX_SRC sources


@pytest.mark.parametrize("chans,cout", [([14, 14], 7), ([28, 28, 1], 64), ([56, 56, 1], 24)])
def test_tc_conv_concatenated_sources(chans, cout):
    """cat(srcs) is never materialised: one TMA tensor map per source, channel blocks staged in groups."""
    from ctunet_b200.engine import Engine
    n, d, h, w, k = 1, 4, 16, 16, 3
    g = torch.Generator().manual_seed(sum(chans))
    xs = [_bf(torch.randn(n, c, d, h, w, generator=g)) for c in chans]
    cin = sum(chans)
    wt = torch.randn(cout, cin, k, k, k, generator=g) / (cin * k ** 3) ** 0.5
    dy = _bf(torch.randn(n, cout, d, h, w, generator=g))
    xr = [x.clone().requires_grad_() for x in xs]
    wr = _bf(wt).requires_grad_()
    yr = F.conv3d(torch.cat(xr, 1), wr, None, 1, 1)
    yr.backward(dy)
    eng = Engine(torch.device(DEV), "bf16", record=True)
    acts = [eng.pack(x.to(DEV)) for x in xs]
    wg = wt.to(DEV).requires_grad_()
    assert eng._tc_ok(k, acts, cout)
    y = eng.conv(acts, wg, None, k, [True] * len(acts), bn_stats=True)
    yo = eng.unpack(y).cpu()
    _check_elementwise(yo, torch.cat(xs, 1), _bf(wt), None, k, "fprop %s -> %d" % (chans, cout))
    cpad = (cout + 7) // 8 * 8
    assert torch.allclose(y.sums.cpu()[:cout], yo.double().sum((0, 2, 3, 4)), rtol=1e-4, atol=1e-2 * yr.abs().max().item())
    assert torch.allclose(y.sums.cpu()[cpad:cpad + cout], (yo.double() ** 2).sum((0, 2, 3, 4)), rtol=1e-4, atol=1e-3)
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    wd = _dgrad_weights(_bf(wt))
    c0 = 0
    for i, a in enumerate(acts):
        dx = eng.unpack(eng.agrads[id(a)]).cpu()
        _check_elementwise(dx, dy, wd[c0:c0 + chans[i]], None, k, "dgrad %s -> %d, source %d" % (chans, cout, i))
        c0 += chans[i]
    dw = eng.pgrads[id(wg)].cpu()
    assert (dw - wr.grad).abs().max().item() <= 2e-3 * wr.grad.abs().max().item()
