"""Per-kernel parity tests (GPU): every C-ABI stage against plain fp32 PyTorch on the CPU.

fp32 'accumulate-check' mode must agree to 1e-4 (north_star); bf16 mode is compared on bf16-rounded
inputs so only the accumulation order and the final bf16 rounding of the output differ.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _eng(mode, record=True):
    from ctunet_b200.engine import Engine
    return Engine(torch.device(DEV), mode, record)


def _tol(mode):
    return dict(rtol=1e-4, atol=1e-4) if mode == "fp32" else dict(rtol=2e-2, atol=2e-2)


def _rnd(mode, t):
    return t if mode == "fp32" else t.to(torch.bfloat16).to(torch.float32)


def _close(a, b, mode, scale=None, what=""):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    ref = b.abs().max().item() if scale is None else scale
    err = (a - b).abs().max().item()
    lim = (1e-4 if mode == "fp32" else 1.2e-2) * max(ref, 1e-6)
    assert err <= lim, "%s: max abs err %.3e > %.3e (ref max %.3e)" % (what, err, lim, ref)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(2, 7, 8, 8, 8), (1, 13, 4, 6, 10), (1, 3, 2, 2, 2)])
def test_pack_unpack_roundtrip(mode, shape):
    g = torch.Generator().manual_seed(0)
    x = _rnd(mode, torch.randn(*shape, generator=g))
    eng = _eng(mode, False)
    a = eng.pack(x.to(DEV))
    assert tuple(a.buf.shape) == (shape[0], (shape[1] + 7) // 8, shape[2], shape[3], shape[4], 8)
    # pad lanes must be zero
    flat = a.buf.float().permute(0, 1, 5, 2, 3, 4).reshape(shape[0], -1, *shape[2:])
    assert torch.equal(flat[:, :shape[1]].cpu(), x)
    assert float(flat[:, shape[1]:].abs().sum()) == 0.0
    assert torch.equal(eng.unpack(a).cpu(), x)


CONV_CASES = [
    # (k, src channels, cout, bias, (n, d, h, w))
    (3, [2], 7, False, (2, 8, 8, 8)),
    (3, [7], 7, False, (1, 16, 16, 16)),
    (3, [28], 7, False, (1, 8, 12, 20)),
    (3, [14, 14], 9, True, (1, 6, 6, 10)),
    (5, [2], 7, True, (1, 8, 8, 8)),
    (5, [8], 16, True, (1, 4, 8, 12)),
    (1, [7, 7], 3, True, (2, 4, 4, 4)),
    (3, [56], 56, False, (1, 2, 2, 2)),
    (3, [3], 5, False, (1, 5, 7, 9)),
]


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv3d_fwd_bwd(mode, case):
    k, chans, cout, use_bias, (n, d, h, w) = case
    g = torch.Generator().manual_seed(1)
    xs = [_rnd(mode, torch.randn(n, c, d, h, w, generator=g)) for c in chans]
    cin = sum(chans)
    wt = torch.randn(cout, cin, k, k, k, generator=g) / (cin * k ** 3) ** 0.5
    bs = torch.randn(cout, generator=g) if use_bias else None
    dy = _rnd(mode, torch.randn(n, cout, d, h, w, generator=g))
    # reference
    xr = [x.clone().requires_grad_() for x in xs]
    wr = wt.clone().requires_grad_()
    br = bs.clone().requires_grad_() if use_bias else None
    yr = F.conv3d(torch.cat(xr, 1), wr, br, 1, k // 2)
    yr.backward(dy)
    # ours
    eng = _eng(mode)
    wg = wt.to(DEV).requires_grad_()
    bg = bs.to(DEV).requires_grad_() if use_bias else None
    acts = [eng.pack(x.to(DEV)) for x in xs]
    y = eng.conv(acts, wg, bg, k, [True] * len(acts))
    _close(eng.unpack(y), yr, mode, what="fprop")
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    for a, x in zip(acts, xr):
        _close(eng.unpack(eng.agrads[id(a)]), x.grad, mode, what="dgrad")
    _close(eng.pgrads[id(wg)], wr.grad, mode, what="wgrad")
    if use_bias:
        _close(eng.pgrads[id(bg)], br.grad, mode, what="dbias")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("case", [([56], (1, 2, 2, 2)), ([7, 7], (2, 4, 4, 4)), ([28, 28], (1, 4, 6, 8)),
                                  ([3], (1, 3, 5, 7))])
def test_convt_fwd_bwd(mode, case):
    chans, (n, d, h, w) = case
    cin = sum(chans)
    g = torch.Generator().manual_seed(2)
    xs = [_rnd(mode, torch.randn(n, c, d, h, w, generator=g)) for c in chans]
    wt = torch.randn(cin, cin, 2, 2, 2, generator=g) / cin ** 0.5
    bs = torch.randn(cin, generator=g)
    dy = _rnd(mode, torch.randn(n, cin, 2 * d, 2 * h, 2 * w, generator=g))
    xr = [x.clone().requires_grad_() for x in xs]
    wr, br = wt.clone().requires_grad_(), bs.clone().requires_grad_()
    yr = F.conv_transpose3d(torch.cat(xr, 1), wr, br, stride=2)
    yr.backward(dy)
    eng = _eng(mode)
    wg, bg = wt.to(DEV).requires_grad_(), bs.to(DEV).requires_grad_()
    acts = [eng.pack(x.to(DEV)) for x in xs]
    y = eng.convt(acts, wg, bg, [True] * len(acts))
    _close(eng.unpack(y), yr, mode, what="convT fprop")
    eng.agrads[id(y)] = eng.pack(dy.to(DEV))
    eng.run_tape()
    for a, x in zip(acts, xr):
        _close(eng.unpack(eng.agrads[id(a)]), x.grad, mode, what="convT dgrad")
    _close(eng.pgrads[id(wg)], wr.grad, mode, what="convT wgrad")
    _close(eng.pgrads[id(bg)], br.grad, mode, what="convT dbias")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("pool", [False, True])
@pytest.mark.parametrize("shape", [(2, 7, 4, 4, 8), (1, 14, 8, 6, 4), (3, 9, 2, 2, 2)])
def test_bn_relu_pool_fwd_bwd(mode, pool, shape):
    n, c, d, h, w = shape
    g = torch.Generator().manual_seed(3)
    x = _rnd(mode, torch.randn(*shape, generator=g) * 1.5 + 0.3)
    bn_ref = torch.nn.BatchNorm3d(c)
    with torch.no_grad():
        bn_ref.weight.copy_(torch.rand(c, generator=g) + 0.5)
        bn_ref.bias.copy_(torch.randn(c, generator=g) * 0.2)
    bn_gpu = torch.nn.BatchNorm3d(c)
    bn_gpu.load_state_dict(bn_ref.state_dict())
    bn_gpu.to(DEV)
    xr = x.clone().requires_grad_()
    ar = F.relu(bn_ref(xr))
    outs_r = [ar]
    if pool:
        outs_r.append(F.max_pool3d(ar, 2, 2))
    gr = [_rnd(mode, torch.randn(o.shape, generator=g)) for o in outs_r]
    torch.autograd.backward(outs_r, gr)

    eng = _eng(mode)
    y = eng.pack(x.to(DEV))
    res = eng.bn_relu(y, bn_gpu, True, extra_updates=1, pool=pool)
    res = res if pool else (res,)
    ss = res[0].bn["ss"].clone()            # the fp32 scale / shift / mean / invstd the kernels use
    for o, r, nm in zip(res, outs_r, ["a", "pooled"]):
        _close(eng.unpack(o), r, mode, what=nm)
    # running stats after the forward update
    assert torch.allclose(bn_gpu.running_mean.cpu(), bn_ref.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(bn_gpu.running_var.cpu(), bn_ref.running_var, rtol=1e-4, atol=1e-5)
    assert int(bn_gpu.num_batches_tracked) == 1
    for o, gg in zip(res, gr):
        eng.agrads[id(o)] = eng.pack(gg.to(DEV))
    eng.run_tape()
    if mode == "bf16" and pool:
        # the routing of every window against float64 with the kernel's fp32 scale / shift: exact, except at windows
        # whose arg-max lies within fp32 rounding of flipping (either child is accepted there; counted)
        import norm_head_oracle as NO
        cpad = (c + 7) // 8 * 8
        ss4 = tuple(ss.double().view(4, cpad)[:, :c].cpu())
        dyo = eng.unpack(eng.agrads[id(y)]).cpu()
        ref, err, gate, tie = NO.dy_error_with_ties(x, ss4, gr[0], gr[1], None, dyo)
        print("tie-marked: %d gates, %d windows" % (int(gate.sum()), int(tie.sum())))
        assert float(err.max()) <= 1.2e-2 * float(ref["dy"].abs().max()), "dy: max abs err %.3e" % float(err.max())
    else:
        _close(eng.unpack(eng.agrads[id(y)]), xr.grad, mode, what="dy")
    _close(eng.pgrads[id(bn_gpu.weight)], bn_ref.weight.grad, mode, what="dgamma")
    _close(eng.pgrads[id(bn_gpu.bias)], bn_ref.bias.grad, mode, what="dbeta")
    # checkpoint quirk: one more update with the same batch statistics happened at backward time
    with torch.no_grad():
        bn_ref(x)
    assert torch.allclose(bn_gpu.running_mean.cpu(), bn_ref.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(bn_gpu.running_var.cpu(), bn_ref.running_var, rtol=1e-4, atol=1e-5)
    assert int(bn_gpu.num_batches_tracked) == 2


def test_bn_eval_mode_uses_running_stats():
    g = torch.Generator().manual_seed(4)
    c = 7
    x = torch.randn(2, c, 4, 4, 4, generator=g)
    bn = torch.nn.BatchNorm3d(c)
    with torch.no_grad():
        bn.running_mean.copy_(torch.randn(c, generator=g) * 0.1)
        bn.running_var.copy_(torch.rand(c, generator=g) + 0.5)
        bn.weight.copy_(torch.rand(c, generator=g) + 0.5)
    bn.eval()
    ref = F.relu(bn(x))
    eng = _eng("fp32", False)
    bg = torch.nn.BatchNorm3d(c)
    bg.load_state_dict(bn.state_dict())
    bg.to(DEV).eval()
    a = eng.bn_relu(eng.pack(x.to(DEV)), bg, False)
    _close(eng.unpack(a), ref, "fp32", what="eval bn")
    assert int(bg.num_batches_tracked) == 0


def _head_ref(xs, w, b, flags):
    from ctunet_b200 import _lib as L
    lc = F.conv3d(torch.cat(xs, 1), w, b)
    out = F.softmax(lc, 1) if flags & L.HEAD_SOFTMAX else lc
    out = torch.sigmoid(out) if flags & L.HEAD_SIGMOID else out
    if flags & (L.HEAD_SP | L.HEAD_SP_SOFTMAX):
        sk = torch.cat((out[:, 0:1], out[:, 1:2] + out[:, 2:3]), 1)
        fl = torch.cat((1 - out[:, 1:2], out[:, 1:2]), 1)
        if flags & L.HEAD_SP_SOFTMAX:
            return F.softmax(sk, 1), F.softmax(fl, 1)
        return sk, fl
    return (out,)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("cfg", [([7, 7], 3, 2 | 4), ([4, 4], 3, 2 | 8), ([8, 8], 2, 1), ([7, 7], 2, 1),
                                 ([8, 8], 2, 2), ([5], 4, 1 | 2), ([16, 16], 2, 0)])
def test_head_fwd_bwd(mode, cfg):
    chans, cout, flags = cfg
    n, d, h, w = 2, 4, 6, 8
    g = torch.Generator().manual_seed(5)
    xs = [_rnd(mode, torch.randn(n, c, d, h, w, generator=g)) for c in chans]
    wt = torch.randn(cout, sum(chans), 1, 1, 1, generator=g) * 0.3
    bs = torch.randn(cout, generator=g) * 0.1
    xr = [x.clone().requires_grad_() for x in xs]
    wr, br = wt.clone().requires_grad_(), bs.clone().requires_grad_()
    outs_r = _head_ref(xr, wr, br, flags)
    gr = [torch.randn(o.shape, generator=g) for o in outs_r]
    torch.autograd.backward(outs_r, gr)
    eng = _eng(mode)
    wg, bg = wt.to(DEV).requires_grad_(), bs.to(DEV).requires_grad_()
    acts = [eng.pack(x.to(DEV)) for x in xs]
    outs = eng.head(acts, wg, bg, flags)
    outs = outs if isinstance(outs, tuple) else (outs,)
    for o, r in zip(outs, outs_r):
        _close(o, r, "fp32", what="head out")       # fp32 math on identical inputs in both modes
    gg = [t.to(DEV) for t in gr]
    eng.backward(gg[0], gg[1] if len(gg) > 1 else None)
    for a, x in zip(acts, xr):
        _close(eng.unpack(eng.agrads[id(a)]), x.grad, mode, what="head dsrc")
    _close(eng.pgrads[id(wg)], wr.grad, "fp32", what="head dw")
    _close(eng.pgrads[id(bg)], br.grad, "fp32", what="head db")


def _dice_ref(p, t):
    b = t.size(0)
    num = (p.reshape(b, -1) * t.reshape(b, -1)).sum(1)
    den = (p.reshape(b, -1) ** 2).sum(1) + (t.reshape(b, -1) ** 2).sum(1)
    return 1 - 2 * torch.mean((num + 1e-7) / (den + 1e-7))


@pytest.mark.parametrize("softmax_for_dice", [True, False])
@pytest.mark.parametrize("c", [2, 3])
def test_dice_ce_fwd_bwd(softmax_for_dice, c):
    from ctunet_b200.losses import dice_ce
    g = torch.Generator().manual_seed(6)
    b, d, h, w = 3, 6, 10, 12
    pred = torch.rand(b, c, d, h, w, generator=g)
    lab = torch.randint(0, c, (b, d, h, w), generator=g)
    tgt = F.one_hot(lab, c).permute(0, 4, 1, 2, 3).float().contiguous()
    pr = pred.clone().requires_grad_()
    ce_r = F.cross_entropy(pr, torch.argmax(tgt, 1))
    dice_r = _dice_ref(F.softmax(pr, 1) if softmax_for_dice else pr, tgt)
    (0.7 * ce_r + 1.3 * dice_r).backward()
    pg = pred.to(DEV).requires_grad_()
    ce, dice = dice_ce(pg, tgt.to(DEV), softmax_for_dice, True)
    (0.7 * ce + 1.3 * dice).backward()
    assert float(ce) == pytest.approx(float(ce_r), rel=1e-5)
    assert float(dice) == pytest.approx(float(dice_r), rel=1e-5)
    _close(pg.grad, pr.grad, "fp32", what="dpred")


def test_dice_loss_module_matches_golden(golden):
    from ctunet_b200 import dice_loss
    d = golden["dice"]
    v = dice_loss()(d["p"].to(DEV), d["t"].to(DEV))
    assert float(v) == pytest.approx(d["value"], rel=1e-6)
    with pytest.raises(RuntimeError):
        dice_loss()(d["p"].to(DEV), d["t"].to(DEV).transpose(2, 3))


def test_hard_segm_bit_exact(golden):
    from ctunet_b200 import hard_segm_from_tensor
    h = golden["hard_segm"]
    y = hard_segm_from_tensor(h["x"].to(DEV))
    assert y.dtype == torch.float32 and torch.equal(y.cpu(), h["y"])
    assert torch.equal(hard_segm_from_tensor(h["x"][0].to(DEV)).cpu(), h["y4"])
    g = torch.Generator().manual_seed(7)
    x = torch.randint(0, 3, (2, 3, 8, 8, 8), generator=g).float()     # many ties
    assert torch.equal(hard_segm_from_tensor(x.to(DEV)).cpu(), torch.argmax(x, 1).float())
    assert hard_segm_from_tensor(x.to(DEV), keep_dims=True).shape == (2, 1, 8, 8, 8)


def test_flap_mask_bit_exact(golden):
    from oracle import unet_oracle as O
    import ctunet_b200 as C
    b = golden["blank_patch"]
    img = b["img"]
    m, e = C.blank_patch(img.to(DEV), b["center"], b["size"], "sphere")
    assert torch.equal(m.cpu(), b["masked"]) and torch.equal(e.cpu(), b["extracted"])
    rng = np.random.RandomState(0)
    for shape in ["sphere", "box"]:
        for it in range(6):
            dims = tuple(int(v) for v in rng.randint(5, 40, 3))
            if it >= 3:                       # rows that are a multiple of 16 voxels take the 16-byte vector kernel
                dims = dims[:2] + (16 * int(rng.randint(1, 4)),)
            vol = (rng.rand(*dims) > 0.6).astype(np.uint8)
            center = [int(rng.randint(0, s)) for s in dims]
            size = int(rng.randint(1, 12))
            mo, eo = O.blank_patch(vol, center, size, shape)
            m, e = C.blank_patch(torch.from_numpy(vol).to(DEV), center, size, shape)
            assert np.array_equal(m.cpu().numpy(), mo) and np.array_equal(e.cpu().numpy(), eo)
            assert np.array_equal((m + e).cpu().numpy(), vol)
    s = golden["shape_3d"]
    sph = C.shape_3d((8, 8, 8), 4, (16, 16, 16), "sphere")
    assert sph.dtype == torch.float64 and int((sph == 0).sum()) == s["sphere_zeros"]
    assert int((C.shape_3d((8, 8, 8), 4, (16, 16, 16), "box") == 0).sum()) == s["box_zeros"]


def test_flap_shape_bit_exact():
    """The 'flap' shape (two cylinders + cube) against the golden vectors made by the reference's own shape_3d /
    random_blank_patch over the restated raster_geometry functions, and against the oracle on random cases."""
    import os
    import random
    import ctunet_b200 as C
    from oracle import unet_oracle as O
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "flap_shape_golden.pt"))
    for c in gold["cases"]:
        shp = C.shape_3d(c["center"], c["size"], c["image_size"], "flap", c_diam=c["c_diam"])
        assert shp.dtype == torch.uint8 and int((shp == 0).sum()) == c["zeros"]
        assert np.array_equal(np.packbits(shp.cpu().numpy()), c["packed"].numpy())
    r = gold["random_blank_patch"]
    random.seed(r["seed"])
    np.random.seed(r["seed"])
    m, e = C.random_blank_patch(r["img"].to(DEV), 1, True, p_type="flap")
    assert torch.equal(m.cpu(), r["masked"]) and torch.equal(e.cpu(), r["extracted"])
    ra = gold["random_blank_patch_any"]                    # p_type="random": shape index drawn from all three shapes
    random.seed(ra["seed"])
    np.random.seed(ra["seed"])
    m, e = C.random_blank_patch(r["img"].to(DEV), 1, True)
    assert torch.equal(m.cpu(), ra["masked"]) and torch.equal(e.cpu(), ra["extracted"])
    rng = np.random.RandomState(3)
    for it in range(8):
        dims = tuple(int(v) for v in rng.randint(6, 48, 3))
        if it >= 4:                           # vector kernel
            dims = dims[:2] + (16 * int(rng.randint(1, 4)),)
        vol = (rng.rand(*dims) > 0.5).astype(np.uint8)
        center = [int(rng.randint(0, s)) for s in dims]
        size, c_diam = int(rng.randint(2, 20)), float(rng.uniform(0.3, 5.0))
        mo, eo = O.blank_patch(vol, center, size, "flap", c_diam)
        m, e = C.blank_patch(torch.from_numpy(vol).to(DEV), center, size, "flap", c_diam)
        assert np.array_equal(m.cpu().numpy(), mo) and np.array_equal(e.cpu().numpy(), eo)


def test_encode_flaprec_batch_bit_exact():
    import ctunet_b200 as C
    from oracle import unet_oracle as O
    g = torch.Generator().manual_seed(5)
    for shape, with_atlas in [((2, 16, 16, 16), True), ((3, 8, 24, 32), False), ((1, 32, 32, 32), True)]:
        full = (torch.rand(shape, generator=g) > 0.6).to(torch.uint8)
        flap = full * (torch.rand(shape, generator=g) > 0.5).to(torch.uint8)
        broken = full - flap
        atlas = torch.rand(shape[1:], generator=g) if with_atlas else None
        ref_img, (ref_sk, ref_fl) = O.encode_flaprec_batch(broken, full, flap, atlas)
        img, (sk, fl) = C.encode_flaprec_batch(broken.to(DEV), full.to(DEV), flap.to(DEV),
                                               atlas.to(DEV) if with_atlas else None)
        assert torch.equal(img.cpu(), ref_img) and torch.equal(sk.cpu(), ref_sk) and torch.equal(fl.cpu(), ref_fl)
    with pytest.raises(RuntimeError):
        C.encode_flaprec_batch(full, full, full)           # CPU tensors: no fallback


def test_kth_nonzero_and_count():
    import ctunet_b200 as C
    rng = np.random.RandomState(1)
    for dims in [(16, 20, 24), (33, 17, 65), (4, 4, 4), (64, 64, 64), (40, 128, 96)]:
        vol = (rng.rand(*dims) > 0.8).astype(np.uint8)
        vol[0, 0, 0] = 1
        t = torch.from_numpy(vol).to(DEV)
        nz = np.argwhere(vol > 0)
        assert C.count_nonzero(t) == nz.shape[0]
        for k in [0, nz.shape[0] // 2, nz.shape[0] - 1]:
            assert C.kth_nonzero(t, k).cpu().tolist() == [int(v) for v in nz[k]]
    assert C.count_nonzero(torch.zeros(8, 8, 8, dtype=torch.uint8, device=DEV)) == 0


def test_random_blank_patch_replays_reference_rng():
    import random
    import ctunet_b200 as C
    from oracle import unet_oracle as O
    rng = np.random.RandomState(5)
    img = (rng.rand(16, 20, 24) > 0.7).astype(np.uint8)
    random.seed(1)
    np.random.seed(1)
    m, e = C.random_blank_patch(torch.from_numpy(img).to(DEV), 1, True, p_type="sphere")
    random.seed(1)
    np.random.seed(1)
    random.uniform(0, 1)
    pix = np.argwhere(img > 0)
    center = pix[np.random.choice(pix.shape[0])]
    lo, hi = O.radius_bounds(img.shape)
    size = np.random.randint(lo, hi)
    mo, eo = O.blank_patch(img, center, size, "sphere")
    assert np.array_equal(m.cpu().numpy(), mo) and np.array_equal(e.cpu().numpy(), eo)
    # empty image: returned unchanged with an empty flap
    z = torch.zeros(8, 8, 8, dtype=torch.uint8, device=DEV)
    m, e = C.random_blank_patch(z, 1, True)
    assert int(m.sum()) == 0 and int(e.sum()) == 0


def test_preprocess_matches_oracle():
    from oracle import unet_oracle as O
    from ctunet_b200 import preprocess as P
    hu = O.skull_phantom_hu((40, 48, 56), 3)
    hg = hu.to(DEV)
    assert torch.equal(P.hu_window(hg, -100.0, 1500.0).cpu(), O.hu_window(hu, -100.0, 1500.0))
    assert torch.equal(P.hu_threshold(hg, 300).cpu(), O.hu_threshold(hu, 300))
    odd = O.skull_phantom_hu((7, 9, 11), 4)       # 693 voxels: vector bulk + scalar tail
    assert torch.equal(P.hu_window(odd.to(DEV), 0.0, 800.0).cpu(), O.hu_window(odd, 0.0, 800.0))
    assert torch.equal(P.hu_threshold(odd.to(DEV), 150).cpu(), O.hu_threshold(odd, 150))
    for out in [(20, 24, 28), (32, 32, 32), (50, 61, 70), (40, 48, 56)]:
        bone = O.hu_threshold(hu, 300)
        assert torch.equal(P.resample_nearest(bone.to(DEV), out).cpu(), O.resample_nearest(bone, out))
        f = O.hu_window(hu, -100.0, 1500.0)
        assert torch.equal(P.resample_nearest(f.to(DEV), out).cpu(), O.resample_nearest(f, out))
        tri = P.resample_trilinear(f.to(DEV), out).cpu()
        assert torch.allclose(tri, O.resample_trilinear(f, out), rtol=1e-5, atol=1e-6)
    for n_in, n_out in [(512, 128), (256, 128), (100, 37), (37, 100), (7, 3)]:
        assert np.array_equal(P.nearest_source_index(n_out, n_in).cpu().numpy(), O.nearest_src_index(n_out, n_in))


def test_errors_are_loud():
    import ctunet_b200 as C
    from ctunet_b200 import _lib
    with pytest.raises(RuntimeError):
        C.hard_segm_from_tensor(torch.zeros(1, 2, 4, 4, 4))          # CPU tensor
    with pytest.raises(RuntimeError):
        _lib.call("ctu_pack_ncdhw", None, None, 0, 1, 1, 1, None)     # null pointers -> error code + message
    assert "bad arguments" in _lib.last_error()


def test_encode_flaprec_bits_is_bit_exact():
    """Bit-packed masks (numpy packbits, bitorder='little') -> float image + atlas channel + uint8 label masks: identical to
    the uint8-mask encoding (datasets.py:195-235) and to the oracle's one-hot targets."""
    import numpy as np
    from ctunet_b200.utilities import encode_flaprec_batch, encode_flaprec_bits, pack_mask_bits
    from oracle import unet_oracle as O
    g = torch.Generator().manual_seed(4)
    shp = (2, 8, 12, 16)
    broken, full, flap = ((torch.rand(shp, generator=g) > t).to(torch.uint8) for t in (0.5, 0.4, 0.8))
    atlas = torch.rand(shp[1:], generator=g)
    bits = [pack_mask_bits(m) for m in (broken, full, flap)]
    for m, b in zip((broken, full, flap), bits):
        assert np.array_equal(b.numpy(), np.packbits(m.numpy().reshape(2, -1), axis=1, bitorder="little"))
        assert torch.equal(pack_mask_bits(m.to(DEV)).cpu(), b)
    img, (fm, lm) = encode_flaprec_bits(*[b.to(DEV) for b in bits], shp[1:], atlas.to(DEV))
    ref_img, (ref_sk, ref_fl) = O.encode_flaprec_batch(broken, full, flap, atlas)
    assert torch.equal(img.cpu(), ref_img)
    assert torch.equal(fm.cpu(), full) and torch.equal(lm.cpu(), flap)
    assert torch.equal(torch.stack((1 - fm, fm), 1).float().cpu(), ref_sk)
    img2, _ = encode_flaprec_batch(broken.to(DEV), full.to(DEV), flap.to(DEV), atlas.to(DEV))
    assert torch.equal(img, img2)
    img1, _ = encode_flaprec_bits(*[b.to(DEV) for b in bits], shp[1:])          # one input channel
    assert img1.shape == (2, 1) + shp[1:] and torch.equal(img1[:, 0].cpu(), broken.float())


@pytest.mark.parametrize("name,mode", [("UNetSP", "fp32"), ("UNetSP", "bf16"), ("recAE_v2_fixed", "bf16")])
def test_fused_sliding_window_equals_unfused(name, mode):
    """Patch gather kernel + head-writes-labels (model.predict_labels, BASELINE config 4) against the unfused pipeline of the
    same modules (slice / stack -> forward -> ctu_argmax_channels -> stitch): BIT-identical label volumes, and the direct
    [B,D,H,W] label path equals hard_segm_from_tensor of the forward outputs."""
    import ctunet_b200 as C
    from ctunet_b200 import preprocess as P
    from oracle import unet_oracle as O
    cfg = O.PRESETS[name]
    C.set_compute_dtype(mode)
    torch.manual_seed(0)
    net = getattr(C, name)().to(DEV).eval()
    C.set_compute_dtype("bf16")
    g = torch.Generator().manual_seed(12)
    vol = (torch.rand(cfg.input_channels, 32, 64, 96, generator=g) > 0.7).float().to(DEV)
    a = P.sliding_window_argmax(net, vol, patch=32, batch=4, fused=True)                  # captured patch batches + ragged tail
    a2 = P.sliding_window_argmax(net, vol, patch=32, batch=4, fused=True, graph=False)
    b = P.sliding_window_argmax(net, vol, patch=32, batch=4, fused=False, graph=False)
    assert len(a) == len(b) == (2 if cfg.head != "plain" else 1)
    for u, u2, v in zip(a, a2, b):
        assert u.shape == (32, 64, 96) and u.dtype == torch.float32
        assert torch.equal(u, v) and torch.equal(u2, v)
    vol2 = vol.flip(3).contiguous()                                                       # a second volume through the same capture
    for u, v in zip(P.sliding_window_argmax(net, vol2, patch=32, batch=4), P.sliding_window_argmax(net, vol2, patch=32, batch=4,
                                                                                             fused=False, graph=False)):
        assert torch.equal(u, v)
    x = torch.stack([vol[:, :, :32, :32], vol[:, :, 32:, 64:]]).contiguous()
    labs = net.predict_labels(x)
    with torch.no_grad():
        out = net(x)
    out = out if isinstance(out, tuple) else (out,)
    for lab, o in zip(labs, out):
        assert torch.equal(lab, C.hard_segm_from_tensor(o))


def test_weight_gather_equals_packing_chain():
    """Weight images produced by the batched index gather (engine._kernel_weights -> ctu_gather_batch) are bit-identical to the
    chain of packing launches whose permutation they replay -- forward and data-gradient variants of the CUDA-core layout
    (tc 0), the resident-weights tcgen05 image (tc 1) and the weight-streaming image (tc 2), single and concatenated sources."""
    from ctunet_b200.engine import Engine, tc_variant
    eng = Engine(torch.device(DEV), "bf16", record=False)
    cases = [
        (7, 3, [2], (2, 32, 32, 32)),
        (14, 3, [7, 7], (1, 32, 32, 32)),
        (64, 3, [14, 14, 1], (1, 16, 16, 16)),        # composed up-stage weights: 8 phases x 8 output channels
        (56, 3, [56], (4, 16, 16, 16)),               # weight-streaming kernel
        (8, 5, [1], (1, 32, 32, 32)),
        (64, 5, [64], (2, 8, 8, 8)),
        (5, 3, [3], (1, 12, 20, 20)),                 # not covered by the tensor paths: packed fp32
    ]
    torch.manual_seed(5)
    seen = set()
    for cout, k, chans, dims in cases:
        native = torch.randn(cout, sum(chans), k, k, k, device=DEV)
        variants = [(None, tc_variant(k, chans, cout, *dims))]
        variants += [((i, c), tc_variant(k, [cout], c, *dims)) for i, c in enumerate(chans)]
        outs = []
        for dgrad_of, tc in variants:
            seen.add(tc)
            want = eng._kernel_weights_chain(native, cout, k, chans, tc, dgrad_of, dims)
            got = eng._kernel_weights(native, cout, k, chans, tc, dgrad_of, dims)
            outs.append((want, got))
        eng._flush_gathers()                           # ONE launch for all variants of the layer
        for want, got in outs:
            assert want.dtype == got.dtype and want.shape == got.shape
            assert torch.equal(want, got)
    assert seen == {0, 1, 2}


def test_accum_prezeroed_flag_matches_library_memset():
    """CTU_ACCUM_PREZEROED (include/ctunet_b200.h): with the flag the entry points ADD into accumulators the caller zeroed
    and enqueue no memset of their own; the sums equal those of the plain calls bit for bit where the reduction order is
    fixed (ctu_bn_stats) and to rounding where atomics commute (fused conv statistics, backward reduction)."""
    from ctunet_b200 import _lib
    from ctunet_b200._lib import CTU_ACCUM_PREZEROED, call, int_array, ptr_array, stream_ptr
    lib = _lib.load()
    eng = _eng("bf16")
    torch.manual_seed(11)
    n, c, d, h, w = 2, 7, 16, 32, 32
    cpad = 8
    x = eng.pack(torch.randn(n, c, d, h, w, device=DEV))
    # ctu_bn_stats
    s_plain = torch.full((2 * cpad,), 123.0, dtype=torch.float64, device=DEV)      # garbage: the call must zero it
    s_flag = torch.zeros(2 * cpad, dtype=torch.float64, device=DEV)
    call("ctu_bn_stats", eng.dtype, x.ptr, c, 1, n, x.spatial, s_plain.data_ptr(), stream_ptr())
    call("ctu_bn_stats", eng.dtype, x.ptr, c, 1 | CTU_ACCUM_PREZEROED, n, x.spatial, s_flag.data_ptr(), stream_ptr())
    assert torch.allclose(s_plain, s_flag, rtol=1e-12, atol=1e-9)
    # the flag really skips the memset: a second flagged call accumulates on top
    call("ctu_bn_stats", eng.dtype, x.ptr, c, 1 | CTU_ACCUM_PREZEROED, n, x.spatial, s_flag.data_ptr(), stream_ptr())
    assert torch.allclose(2 * s_plain, s_flag, rtol=1e-12, atol=1e-9)
    # fused statistics of the tcgen05 convolution
    wt = torch.randn(7, c, 3, 3, 3, device=DEV) * 0.1
    wk = eng._kernel_weights_chain(wt, 7, 3, [c], 1)
    y = eng.new_act(7, n, d, h, w)
    sums = []
    for flag, init in ((0, 55.0), (CTU_ACCUM_PREZEROED, 0.0)):
        s = torch.full((2 * cpad,), init, dtype=torch.float64, device=DEV)
        call("ctu_conv3d_fprop", eng.dtype, ptr_array([x.ptr]), int_array([c]), 1, wk.data_ptr(), None, y.ptr, s.data_ptr(), 0,
             7, 3, n, d, h, w, 1 | flag, stream_ptr())
        sums.append(s)
    assert torch.allclose(sums[0], sums[1], rtol=1e-9, atol=1e-6)
    # BatchNorm backward reduction
    ss = torch.rand(4 * cpad, device=DEV)
    dA = eng.pack(torch.randn(n, c, d, h, w, device=DEV))
    red = []
    for flag, init in ((0, -7.0), (CTU_ACCUM_PREZEROED, 0.0)):
        s = torch.full((2 * cpad,), init, dtype=torch.float64, device=DEV)
        call("ctu_bn_relu_bwd_reduce", eng.dtype, x.ptr, ss.data_ptr(), dA.ptr, None, s.data_ptr(), c, n, d, h, w, 0 | flag, stream_ptr())
        red.append(s)
    assert torch.allclose(red[0], red[1], rtol=1e-9, atol=1e-6)
