"""Random affine augmentation on the GPU (csrc/augment.cu): the fused encoder and the mask gather bit for bit against the
CPU oracle (tests/affine_oracle.py), the draws bit for bit against the numpy Philox restatement, their statistics, the
random state, and TrainStep(augment=...) eager and captured against the plain step fed the transformed masks."""
import numpy as np
import pytest
import torch

import affine_oracle as A

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _skull_batch(b, shape, seed):
    """(broken, full, flap) uint8 [B, D, H, W] with broken & flap == 0, broken | flap == full (CPU numpy)."""
    g = np.random.default_rng(seed)
    d, h, w = shape
    zz, yy, xx = np.meshgrid(*[np.linspace(-1, 1, n) for n in shape], indexing="ij")
    out = []
    for i in range(b):
        r = np.sqrt((zz / 0.8) ** 2 + (yy / 0.85) ** 2 + (xx / 0.7) ** 2) + 0.02 * g.standard_normal(shape)
        full = ((r > 0.8) & (r <= 1.0)).astype(np.uint8) | (g.random(shape) < 0.01).astype(np.uint8)
        c = g.uniform(-0.5, 0.5, 3)
        flap = full & (((zz - c[0]) ** 2 + (yy - c[1]) ** 2 + (xx - c[2]) ** 2) < 0.2).astype(np.uint8)
        out.append((full - flap, full, flap))
    return [np.stack([o[k] for o in out]) for k in range(3)]


def _random_matrices(b, shape, seed, rot=30.0, scale=(0.8, 1.25), shift=8.0):
    g = np.random.default_rng(seed)
    p = np.zeros((b, 10))
    p[:, :3] = np.radians(g.uniform(-rot, rot, (b, 3)))
    p[:, 3] = g.uniform(*scale, b)
    p[:, 4:7] = g.uniform(-shift, shift, (b, 3))
    p[:, 7:] = np.where(g.random((b, 3)) < 0.5, -1.0, 1.0)
    return A.matrix_from_params(p.astype(np.float32), shape)


def _encode(bits, srcs, mats, atlas, vol):
    from ctunet_b200 import _lib
    b = mats.shape[0]
    cin = 1 if atlas is None else 2
    image = torch.full((b, cin) + vol, -1.0, device=DEV)
    fm = torch.full((b,) + vol, 7, dtype=torch.uint8, device=DEV)
    lm = torch.full_like(fm, 7)
    _lib.call("ctu_affine_encode_flaprec", bits, *[s.data_ptr() for s in srcs], atlas.data_ptr() if atlas is not None else None,
              mats.data_ptr(), image.data_ptr(), fm.data_ptr(), lm.data_ptr(), b, cin, *vol, _lib.stream_ptr())
    return image, fm, lm


def _ulps(a, b):
    def key(x):
        i = np.asarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


@pytest.mark.parametrize("bits", [0, 1])
@pytest.mark.parametrize("with_atlas", [False, True])
@pytest.mark.parametrize("b,shape", [(4, (128, 128, 128)), (3, (24, 20, 18))])
def test_fused_encoder_matches_oracle(bits, with_atlas, b, shape):
    """Image channel 0, the atlas channel and both label masks bit for bit, for the 16-byte-vector variant (128^3) and the
    voxel-by-voxel one (w = 18), under random rotations up to 30 degrees, scales 0.8-1.25, translations and flips."""
    from ctunet_b200.utilities import pack_mask_bits
    masks = _skull_batch(b, shape, seed=b)
    mats = _random_matrices(b, shape, seed=10 + b)
    mats[0] = A.identity(1)[0]
    ref = A.sample(masks, mats)
    dev = [torch.from_numpy(m).to(DEV) for m in masks]
    srcs = [pack_mask_bits(m) for m in dev] if bits else dev
    atlas = torch.rand(shape, device=DEV) if with_atlas else None
    image, fm, lm = _encode(bits, srcs, torch.from_numpy(mats).to(DEV), atlas, shape)
    assert torch.equal(image[:, 0].cpu(), torch.from_numpy(ref[0]).float())
    if with_atlas:
        assert torch.equal(image[:, 1], atlas.expand(b, *shape))
    assert np.array_equal(fm.cpu().numpy(), ref[1]) and np.array_equal(lm.cpu().numpy(), ref[2])
    assert np.array_equal(ref[1][0], masks[1][0])                          # sample 0: the identity
    br = ref[0].astype(bool)
    assert not np.any(br & ref[2].astype(bool)) and np.array_equal(br | ref[2].astype(bool), ref[1].astype(bool))


@pytest.mark.parametrize("dtype", [torch.uint8, torch.bool])
@pytest.mark.parametrize("n,shape", [(1, (16, 16, 32)), (2, (9, 13, 21)), (3, (20, 24, 16))])
def test_affine_masks_matches_oracle(dtype, n, shape):
    from ctunet_b200 import affine_masks
    masks = _skull_batch(2, shape, seed=n)[:n]
    mats = _random_matrices(2, shape, seed=n)
    out = affine_masks([torch.from_numpy(m).to(DEV).to(dtype) for m in masks], torch.from_numpy(mats).to(DEV))
    for o, r in zip(out, A.sample(masks, mats)):
        assert o.dtype == dtype and tuple(o.shape) == (2,) + shape
        assert np.array_equal(o.cpu().numpy().astype(np.uint8), r)


def test_non_finite_matrices_read_zero():
    from ctunet_b200 import affine_masks
    shape = (8, 8, 16)
    m = torch.ones((4,) + shape, dtype=torch.uint8, device=DEV)
    mats = A.identity(4)
    mats[0, 0, 3] = np.nan
    mats[1, 1, 1] = np.inf
    mats[2, 2, 3] = -np.inf
    mats[3, 2, 2] = np.float32(3e38)
    out = affine_masks([m], torch.from_numpy(mats).to(DEV))[0].cpu().numpy()
    assert np.array_equal(out, A.sample([m.cpu().numpy()], mats)[0])
    assert out[0].sum() == 0 and out[1].sum() == 0 and out[2].sum() == 0
    assert out[3].sum() == out[3, :, :, 0].sum()                       # only x = 0 keeps a finite source


def test_draws_match_numpy_philox_and_matrices():
    from ctunet_b200 import RandomAffine
    ra = RandomAffine(rotate=(20, 10, 30), scale=(0.85, 1.2), translate=(6, 4, 2), flip=(True, False, True))
    vol = (96, 112, 80)
    for pass_ in range(3):
        params, mats = ra.draw(300, vol, DEV)
        key, counter = ra._state[torch.device(DEV, torch.cuda.current_device())]
        assert int(counter) == pass_ + 1
        ref = A.draw(key, pass_, 300, A.ranges_f32(ra.rotate, ra.scale, ra.translate), 0b101)
        assert np.array_equal(params.cpu().numpy(), ref)
        assert _ulps(mats.cpu().numpy(), A.matrix_from_params(ref, vol)).max() <= 1
    assert ra.last[0] is params and ra.last[1] is mats


def test_draw_statistics():
    from ctunet_b200 import RandomAffine
    rot, sc, tr = (15.0, 15.0, 15.0), (0.9, 1.1), (8.0, 8.0, 8.0)
    n = 4096
    params = RandomAffine(rot, sc, tr, (True, True, True)).draw(n, (128, 128, 128), DEV)[0].cpu().numpy()
    for k in range(3):
        r = np.float32(np.radians(rot[k]))
        assert np.abs(params[:, k]).max() <= r
        sigma = r / np.sqrt(3) / np.sqrt(n)
        assert abs(params[:, k].mean()) <= 5 * sigma
        assert np.abs(params[:, 4 + k]).max() <= tr[k]
        flips = (params[:, 7 + k] == -1).sum()
        assert set(np.unique(params[:, 7 + k])) == {-1.0, 1.0}
        assert abs(flips - n / 2) <= 5 * np.sqrt(n / 4)
    assert params[:, 3].min() >= np.float32(sc[0]) and params[:, 3].max() <= np.float32(sc[1])
    # default: only the left-right axis flips
    p = RandomAffine().draw(n, (64, 64, 64), DEV)[0].cpu().numpy()
    assert np.all(p[:, 7:9] == 1) and 0 < (p[:, 9] == -1).sum() < n


def test_random_state_reproduces_and_advances():
    from ctunet_b200 import RandomAffine
    torch.manual_seed(123)
    a = RandomAffine()
    first = [a.draw(4, (32, 32, 32), DEV)[0].clone() for _ in range(3)]
    assert not torch.equal(first[0], first[1]) and not torch.equal(first[1], first[2])
    torch.manual_seed(123)
    b = RandomAffine()
    assert all(torch.equal(f, b.draw(4, (32, 32, 32), DEV)[0]) for f in first)
    torch.manual_seed(124)
    assert not torch.equal(RandomAffine().draw(4, (32, 32, 32), DEV)[0], first[0])


def test_sample_dict_composes_with_skull_random_hole():
    from ctunet_b200 import RandomAffine, SkullRandomHole, affine_masks
    full = torch.from_numpy(_skull_batch(2, (32, 32, 32), 5)[1]).to(DEV)
    s = SkullRandomHole(double_output=True)({"image": full})
    ra = RandomAffine(rotate=20)
    out = ra(s)
    brk, (fu, fl) = out["image"], out["target"]
    ref = affine_masks([s["image"], s["target"][0], s["target"][1]], ra.last[1])
    assert all(torch.equal(x, y) for x, y in zip((brk, fu, fl), ref))
    assert int((brk & fl).sum()) == 0 and torch.equal(brk | fl, fu)
    one = ra({"image": full[0], "target": full[0]})                      # [D, H, W] with a single target
    assert one["image"].shape == full[0].shape and torch.equal(one["image"], one["target"])
    with pytest.raises(ValueError):
        ra({"image": full.float(), "target": full})


def _batch(b, size, seed):
    from ctunet_b200.synthetic import make_training_batch
    from ctunet_b200.utilities import pack_mask_bits
    img, (sk_t, fl_t) = make_training_batch(b, 2, size, seed=seed, device=DEV)
    masks = [t.to(torch.uint8).contiguous() for t in (img[:, 0], sk_t[:, 1], fl_t[:, 1])]
    return masks, [pack_mask_bits(m) for m in masks], img[0, 1].contiguous()


def _net():
    import ctunet_b200 as C
    C.set_compute_dtype("bf16")
    torch.manual_seed(0)
    return C.UNetSP().to(DEV).train()


def test_identity_augmentation_equals_the_plain_encoder_and_step():
    from ctunet_b200 import RandomAffine
    from ctunet_b200.trainer import TrainStep
    from ctunet_b200.utilities import encode_flaprec_batch, encode_flaprec_bits
    masks, bits, atlas = _batch(2, 32, 3)
    vol = tuple(masks[0].shape[1:])
    eye = torch.from_numpy(A.identity(2)).to(DEV)
    ref_img, (ref_fm, ref_lm) = encode_flaprec_bits(*bits, vol, atlas)
    for fmt, srcs in ((1, bits), (0, masks)):
        image, fm, lm = _encode(fmt, srcs, eye, atlas, vol)
        assert torch.equal(image, ref_img) and torch.equal(fm, ref_fm) and torch.equal(lm, ref_lm)
    assert torch.equal(encode_flaprec_batch(*masks, atlas, out=(torch.empty_like(ref_img), None))[0], ref_img)
    ident = RandomAffine(0, (1, 1), 0, (False, False, False))
    plain, aug = TrainStep(_net(), "double", lr=1e-5), TrainStep(_net(), "double", lr=1e-5, augment=ident)
    for _ in range(2):
        a = plain.step_from_bits(*bits, vol, atlas).tolist()
        b = aug.step_from_bits(*bits, vol, atlas).tolist()
        assert a == pytest.approx(b, rel=2e-3, abs=2e-3)
    assert torch.equal(aug.last_affine()[1], eye)


@pytest.mark.parametrize("graph", [False, True])
def test_augmented_step_equals_plain_step_on_transformed_masks(graph):
    """TrainStep(augment=...).step_from_bits against a plain TrainStep.step_from_masks fed affine_masks(masks, the matrices
    the augmenting step drew), two identically initialised UNetSP: same encoder outputs bit for bit, loss components and
    parameters within the tolerances of the eager-versus-graph step test."""
    from ctunet_b200 import RandomAffine, affine_masks
    from ctunet_b200.trainer import TrainStep
    from ctunet_b200.utilities import encode_flaprec_batch
    masks, bits, atlas = _batch(2, 32, 4)
    vol = tuple(masks[0].shape[1:])
    net_a, net_p = _net(), _net()
    torch.manual_seed(7)
    aug = TrainStep(net_a, "double", lr=1e-5, graph=graph, augment=RandomAffine(rotate=20, translate=4))
    plain = TrainStep(net_p, "double", lr=1e-5, graph=graph)
    drawn = []
    for _ in range(4):
        ca = aug.step_from_bits(*bits, vol, atlas).tolist()
        params, mats = aug.last_affine()
        drawn.append(params.clone())
        tm = affine_masks(masks, mats)
        cp = plain.step_from_masks(*tm, atlas).tolist()
        assert ca == pytest.approx(cp, rel=2e-2, abs=2e-2)
        image, fm, lm = _encode(1, bits, mats, atlas, vol)
        ref_img, _ = encode_flaprec_batch(*tm, atlas, out=(torch.empty_like(image), None))
        assert torch.equal(image, ref_img) and torch.equal(fm, tm[1]) and torch.equal(lm, tm[2])
        if graph and aug._graph is not None:
            assert torch.equal(aug._static[0], image) and torch.equal(aug._static[1], fm)
    assert all(not torch.equal(drawn[i], drawn[i + 1]) for i in range(3))
    if graph:
        assert aug.launches_per_step == plain.launches_per_step
    sa, sp = net_a.state_dict(), net_p.state_dict()
    for k in sa:
        if k.endswith("num_batches_tracked"):
            assert int(sa[k]) == int(sp[k]), k
        elif "running" in k:
            assert torch.allclose(sa[k], sp[k], rtol=5e-2, atol=2e-2 * float(sa[k].abs().max()) + 1e-6), k
        elif not k.startswith("cblock"):
            assert float((sa[k] - sp[k]).abs().max()) <= 1e-4, k


def test_graph_and_eager_augmented_steps_draw_the_same_transforms():
    from ctunet_b200 import RandomAffine
    from ctunet_b200.trainer import TrainStep
    masks, bits, atlas = _batch(2, 32, 5)
    vol = tuple(masks[0].shape[1:])
    hist = []
    for graph in (False, True):
        net = _net()
        torch.manual_seed(11)
        step = TrainStep(net, "double", lr=1e-5, graph=graph, augment=RandomAffine())
        ps, cs = [], []
        for _ in range(5):                                # 2 eager warm-up steps, the capture, 2 replays
            cs.append(step.step_from_masks(*masks, atlas).tolist())
            ps.append(step.last_affine()[0].clone())
        hist.append((ps, cs))
        if graph:
            assert step._graph is not None
    (pe, ce), (pg, cg) = hist
    assert all(torch.equal(a, b) for a, b in zip(pe, pg))
    assert all(not torch.equal(pg[i], pg[i + 1]) for i in range(4))    # fresh transforms on every replay
    for a, b in zip(ce, cg):
        assert a == pytest.approx(b, rel=2e-2, abs=2e-2)


def test_errors_before_any_launch(monkeypatch):
    from ctunet_b200 import RandomAffine, _lib
    from ctunet_b200 import trainer as T
    from ctunet_b200.trainer import TrainStep
    masks, bits, atlas = _batch(2, 32, 6)
    vol = tuple(masks[0].shape[1:])
    step = TrainStep(_net(), "double", lr=1e-5, augment=RandomAffine())
    img = torch.zeros((2, 2) + vol, device=DEV)
    n0 = _lib.launches
    with pytest.raises(ValueError):
        step(img, (masks[1], masks[2]))                                      # a ready float image
    with pytest.raises(TypeError):
        step.step_from_masks(masks[0].float(), masks[1], masks[2], atlas)
    with pytest.raises(RuntimeError):
        step.step_from_masks(masks[0].cpu(), masks[1], masks[2], atlas)
    with pytest.raises(ValueError):
        step.step_from_bits(*bits, (32, 32, 16), atlas)
    with pytest.raises(TypeError):
        step.step_from_bits(*bits, vol, atlas.double())
    with pytest.raises(TypeError):
        TrainStep(_net(), "double", augment=object())
    monkeypatch.setattr(T, "FUSED_HEAD_LOSS", False)
    with pytest.raises(ValueError):
        step.step_from_masks(*masks, atlas)                                  # float one-hot targets
    from ctunet_b200 import affine_masks
    with pytest.raises(ValueError):
        affine_masks(masks, torch.zeros(2, 3, 3, device=DEV))
    with pytest.raises(ValueError):
        affine_masks(masks, torch.zeros(2, 3, 4, device=DEV, dtype=torch.float64))
    with pytest.raises(RuntimeError):
        affine_masks(masks, torch.zeros(2, 3, 4))
    assert _lib.launches == n0
    assert step.last_affine() is None
