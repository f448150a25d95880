"""The virtual craniectomy on the GPU (csrc/augment.cu, DESIGN.md section 7f): the draws bit for bit against the CPU oracle
(tests/craniectomy_oracle.py), the fused encoder with and without RandomAffine bit for bit against the oracle and against
affine_masks(blank_patch(...)), the draw statistics, the random state and the absence of host synchronisation, and
TrainStep(craniectomy=...) eager and captured against a plain step fed the oracle's masks."""
import numpy as np
import pytest
import torch

import affine_oracle as A
import craniectomy_oracle as K

pytestmark = pytest.mark.gpu

DEV = "cuda"
ODD = (24, 56, 72)                         # w % 16 != 0: the voxel-by-voxel encoder


def _skulls(b, shape, seed):
    """Full-skull-like uint8 masks [B, D, H, W] (CPU numpy): a noisy ellipsoidal shell plus sparse voxels."""
    g = np.random.default_rng(seed)
    zz, yy, xx = np.meshgrid(*[np.linspace(-1, 1, n) for n in shape], indexing="ij")
    out = []
    for _ in range(b):
        r = np.sqrt((zz / 0.8) ** 2 + (yy / 0.85) ** 2 + (xx / 0.7) ** 2) + 0.02 * g.standard_normal(shape)
        out.append(((r > 0.8) & (r <= 1.0)).astype(np.uint8) | (g.random(shape) < 0.005).astype(np.uint8))
    return np.stack(out)


def _key(rc):
    return rc._state[torch.device(DEV, torch.cuda.current_device())]


def _rows(full, seed):
    """Hand-made params: sample b gets shape b % 3 about a bone voxel, the last sample is not applied."""
    g = np.random.default_rng(seed)
    b_, vol = full.shape[0], full.shape[1:]
    min_r, max_r = K.radius_bounds(vol)
    rows = np.zeros((b_, 7))
    for b in range(b_):
        bone = np.argwhere(full[b] > 0)
        radius = int(g.integers(min_r, max_r))
        shape = b % 3
        c_diam = (0.25 + 0.75 * g.random()) * radius / 4 if shape == 2 else 0.0
        rows[b] = [float(b != b_ - 1 or b_ == 1), shape, radius, c_diam] + list(bone[g.integers(len(bone))])
    return rows


@pytest.mark.parametrize("bits", [0, 1])
@pytest.mark.parametrize("b,shape", [(1, ODD), (4, (128, 128, 128)), (7, ODD)])
@pytest.mark.parametrize("shapes", [("sphere",), ("box",), ("flap",), ("sphere", "box", "flap")])
def test_draws_match_oracle(bits, b, shape, shapes):
    from ctunet_b200 import RandomCraniectomy
    from ctunet_b200.utilities import pack_mask_bits
    full = _skulls(b, shape, seed=b)
    if b == 7:
        full[3] = 0                                                       # an empty skull: no hole, counter still advances
    dev = torch.from_numpy(full).to(DEV)
    src = pack_mask_bits(dev) if bits else dev
    rc = RandomCraniectomy(1.0, shapes)
    for pass_ in range(2):
        params = rc.draw(src, shape if bits else None)
        key, counter = _key(rc)
        assert int(counter) == pass_ + 1
        ref = K.draw(key, pass_, full, 1.0, shapes)
        assert np.array_equal(params.cpu().numpy(), ref), (pass_, params.cpu().numpy(), ref)
        assert rc.last is params
    if b == 7:
        assert ref[3, 0] == 0 and tuple(ref[3, 4:]) == (-1, -1, -1)
    assert set(np.unique(ref[:, 1]).astype(int)) <= {K.SHAPE_CODES[s] for s in shapes}


@pytest.mark.parametrize("p", [1.0, 0.5, 0.0])
def test_gate_matches_oracle(p):
    from ctunet_b200 import RandomCraniectomy
    full = _skulls(7, ODD, seed=11)
    rc = RandomCraniectomy(p)
    for pass_ in range(3):
        params = rc.draw(torch.from_numpy(full).to(DEV)).cpu().numpy()
        assert np.array_equal(params, K.draw(_key(rc)[0], pass_, full, p))
    if p == 0.0:
        assert np.all(params[:, 0] == 0)
    broken, f, flap = (t.cpu().numpy() for t in _masks_u8(torch.from_numpy(full).to(DEV), torch.from_numpy(params).to(DEV)))
    assert all(np.array_equal(x, y) for x, y in zip((broken, f, flap), K.cut(full, params)))


def _masks_u8(full, params):
    from ctunet_b200 import _lib
    b, d, h, w = full.shape
    out = [torch.full_like(full, 7) for _ in range(3)]
    _lib.call("ctu_craniectomy_masks_u8", full.data_ptr(), params.data_ptr(), *[t.data_ptr() for t in out], b, d, h, w,
              _lib.stream_ptr())
    return out


def _encode(bits, src, params, mats, atlas, vol):
    from ctunet_b200 import _lib
    b = params.shape[0]
    cin = 1 if atlas is None else 2
    image = torch.full((b, cin) + vol, -1.0, device=DEV)
    fm = torch.full((b,) + vol, 7, dtype=torch.uint8, device=DEV)
    lm = torch.full_like(fm, 7)
    _lib.call("ctu_craniectomy_encode_flaprec", bits, src.data_ptr(), params.data_ptr(),
              atlas.data_ptr() if atlas is not None else None, mats.data_ptr() if mats is not None else None, image.data_ptr(),
              fm.data_ptr(), lm.data_ptr(), b, cin, *vol, _lib.stream_ptr())
    return image, fm, lm


def _random_matrices(b, shape, seed):
    g = np.random.default_rng(seed)
    p = np.zeros((b, 10))
    p[:, :3] = np.radians(g.uniform(-30, 30, (b, 3)))
    p[:, 3] = g.uniform(0.8, 1.25, b)
    p[:, 4:7] = g.uniform(-8, 8, (b, 3))
    p[:, 7:] = np.where(g.random((b, 3)) < 0.5, -1.0, 1.0)
    return A.matrix_from_params(p.astype(np.float32), shape)


@pytest.mark.parametrize("bits", [0, 1])
@pytest.mark.parametrize("with_atlas", [False, True])
@pytest.mark.parametrize("affine", [False, True])
@pytest.mark.parametrize("b,shape", [(4, (128, 128, 128)), (4, ODD)])
def test_encoder_matches_oracle(bits, with_atlas, affine, b, shape):
    """Image channel 0 (broken), the atlas channel and both label masks bit for bit, for sphere, box, flap and a sample
    that is not applied; with RandomAffine matrices also against affine_masks(blank_patch(...)) on the device."""
    from ctunet_b200 import affine_masks, blank_patch
    from ctunet_b200.utilities import pack_mask_bits
    full = _skulls(b, shape, seed=20 + b)
    rows = _rows(full, seed=b)
    mats = _random_matrices(b, shape, seed=30 + b) if affine else None
    ref = K.encode(full, rows, mats)
    dev = torch.from_numpy(full).to(DEV)
    src = pack_mask_bits(dev) if bits else dev
    atlas = torch.rand(shape, device=DEV) if with_atlas else None
    dmats = torch.from_numpy(mats).to(DEV) if affine else None
    image, fm, lm = _encode(bits, src, torch.from_numpy(rows).to(DEV), dmats, atlas, shape)
    assert torch.equal(image[:, 0].cpu(), torch.from_numpy(ref[0]).float())
    if with_atlas:
        assert torch.equal(image[:, 1], atlas.expand(b, *shape))
    assert np.array_equal(fm.cpu().numpy(), ref[1]) and np.array_equal(lm.cpu().numpy(), ref[2])
    br = ref[0].astype(bool)
    assert not np.any(br & ref[2].astype(bool)) and np.array_equal(br | ref[2].astype(bool), ref[1].astype(bool))
    if affine:
        cut = [blank_patch(dev[i], [int(c) for c in rows[i, 4:]], rows[i, 2], K.SHAPE_NAMES[int(rows[i, 1])],
                           rows[i, 3] if rows[i, 1] == 2 else None) if rows[i, 0] else (dev[i], torch.zeros_like(dev[i]))
               for i in range(b)]
        tm = affine_masks([torch.stack([c[0] for c in cut]), dev, torch.stack([c[1] for c in cut])], dmats)
        assert torch.equal(image[:, 0], tm[0].float()) and torch.equal(fm, tm[1]) and torch.equal(lm, tm[2])
    else:
        assert sum(int(lm[i].sum()) > 0 for i in range(b - 1)) == b - 1       # every applied hole removed bone


def _draw_abi(bits, src, batch, vol, p, key, pass_counter):
    """ctu_craniectomy_draw straight through the C ABI (any bit stream, also one whose volume is not a whole byte)."""
    from ctunet_b200 import _lib
    min_r, max_r = K.radius_bounds(vol)
    nbytes = _lib.load().ctu_craniectomy_workspace_bytes(batch, *vol)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    params = torch.empty((batch, 7), dtype=torch.float64, device=DEV)
    _lib.call("ctu_craniectomy_draw", bits, src.data_ptr(), batch, *vol, p, 7, min_r, max_r, key, pass_counter.data_ptr(),
              params.data_ptr(), ws.data_ptr(), nbytes, _lib.stream_ptr())
    return params


@pytest.mark.parametrize("case", ["bits_odd_offset", "u8_odd_offset", "bits_stream_not_whole_bytes"])
def test_unaligned_views_and_tail_paths(case):
    """Batches of 37 (> 32: a warp of the draw kernel takes two samples) whose volumes are not a multiple of 32 voxels,
    read through views that start at odd byte addresses: the per-byte paths of the count kernel, of bone_word and of the
    encoder, bit for bit against the oracle, draws and masks (with and without affine matrices)."""
    from ctunet_b200 import RandomCraniectomy
    from ctunet_b200.utilities import pack_mask_bits
    vol = {"bits_odd_offset": (9, 9, 8), "u8_odd_offset": (23, 37, 41), "bits_stream_not_whole_bytes": (3, 5, 7)}[case]
    full = _skulls(38, vol, seed=len(case))
    full[5] = 0                                                           # an empty skull
    full[37] = 0
    full[37].flat[-1] = 1                                                 # bone only in the last voxel of the batch
    host = full[1:]
    if case == "bits_stream_not_whole_bytes":                           # 105 voxels per sample: one bit stream for the batch
        bits, stream = 1, torch.from_numpy(np.packbits(host.ravel(), bitorder="little")).to(DEV)
        key = 0x5EED_0000_0000_0001
        counter = torch.zeros(1, dtype=torch.int64, device=DEV)
        params = [_draw_abi(1, stream, 37, vol, 0.8, key, counter) for _ in range(2)]
        src = stream
    else:
        dev = torch.from_numpy(full).to(DEV)
        bits = int(case.startswith("bits"))
        src = (pack_mask_bits(dev) if bits else dev)[1:]                # odd byte offset: 81 or 34891 bytes per sample
        assert src.data_ptr() % 2 == 1
        rc = RandomCraniectomy(0.8)
        params = [rc.draw(src, vol if bits else None).clone() for _ in range(2)]
        key = _key(rc)[0]
    for pass_, prm in enumerate(params):
        ref = K.draw(key, pass_, host, 0.8)
        assert np.array_equal(prm.cpu().numpy(), ref), pass_
    assert ref[4, 0] == 0 and ref[36, 0] in (0, 1)
    if ref[36, 0]:
        assert tuple(ref[36, 4:]) == tuple(int(v) - 1 for v in vol)
    mats = _random_matrices(37, vol, seed=9)
    for m in (None, mats):
        out = _encode(bits, src, params[1], None if m is None else torch.from_numpy(m).to(DEV), None, vol)
        want = K.encode(host, params[1].cpu().numpy(), m)
        assert torch.equal(out[0][:, 0].cpu(), torch.from_numpy(want[0]).float())
        assert np.array_equal(out[1].cpu().numpy(), want[1]) and np.array_equal(out[2].cpu().numpy(), want[2])


def test_draw_statistics():
    """4096 draws on an 8 x 8 x 64 volume with 10 bone voxels: the centre is uniform over them, the radius over
    [0, 18), the shape over the three; the gate fires at rate p."""
    from scipy.stats import chi2
    from ctunet_b200 import RandomCraniectomy
    n = 4096
    full = np.zeros((n, 8, 8, 64), dtype=np.uint8)
    g = np.random.default_rng(0)
    flat = g.choice(8 * 8 * 64, 10, replace=False)
    full.reshape(n, -1)[:, flat] = 1
    dev = torch.from_numpy(full).to(DEV)
    params = RandomCraniectomy().draw(dev).cpu().numpy()
    assert np.all(params[:, 0] == 1)

    def chi2_ok(counts):
        counts = np.asarray(counts, dtype=np.float64)
        e = counts.sum() / len(counts)
        return chi2.sf(((counts - e) ** 2 / e).sum(), len(counts) - 1) > 1e-4

    vox = np.ravel_multi_index(params[:, 4:].astype(np.int64).T, (8, 8, 64))
    assert set(vox) <= set(flat) and chi2_ok([np.sum(vox == v) for v in flat])
    min_r, max_r = K.radius_bounds((8, 8, 64))
    assert (min_r, max_r) == (0, 18)
    assert params[:, 2].min() >= min_r and params[:, 2].max() < max_r
    assert chi2_ok(np.bincount(params[:, 2].astype(int) - min_r, minlength=max_r - min_r))
    assert chi2_ok(np.bincount(params[:, 1].astype(int), minlength=3))
    flap = params[params[:, 1] == 2]
    lo, hi = 0.25 * flap[:, 2] / 4, flap[:, 2] / 4
    assert np.all((flap[:, 3] >= lo) & (flap[:, 3] <= hi)) and np.all(params[params[:, 1] != 2, 3] == 0)
    for p in (0.3, 0.75):
        applied = RandomCraniectomy(p).draw(dev).cpu().numpy()[:, 0]
        assert abs(applied.mean() - p) <= 5 * np.sqrt(p * (1 - p) / n)


def test_random_state_reproduces_and_advances():
    from ctunet_b200 import RandomCraniectomy
    full = torch.from_numpy(_skulls(4, (32, 32, 32), 1)).to(DEV)
    torch.manual_seed(123)
    a = RandomCraniectomy()
    first = [a.draw(full).clone() for _ in range(3)]
    assert not torch.equal(first[0], first[1]) and not torch.equal(first[1], first[2])
    torch.manual_seed(123)
    b = RandomCraniectomy()
    assert all(torch.equal(f, b.draw(full)) for f in first)
    torch.manual_seed(124)
    assert not torch.equal(RandomCraniectomy().draw(full), first[0])


def test_sample_dict_and_composition_with_random_affine():
    from ctunet_b200 import RandomAffine, RandomCraniectomy, affine_masks
    full = torch.from_numpy(_skulls(3, (32, 32, 48), 5)).to(DEV)
    rc = RandomCraniectomy()
    s = rc({"image": full, "name": "x"})
    assert s["name"] == "x"
    ref = K.cut(full.cpu().numpy(), rc.last.cpu().numpy())
    assert all(np.array_equal(t.cpu().numpy(), r) for t, r in zip((s["image"],) + tuple(s["target"]), ref))
    ra = RandomAffine(rotate=20)
    out = ra(s)
    tm = affine_masks([s["image"], s["target"][0], s["target"][1]], ra.last[1])
    assert all(torch.equal(x, y) for x, y in zip((out["image"],) + tuple(out["target"]), tm))
    one = rc({"image": full[0].bool()})                                   # [D, H, W], bool
    brk, (fu, fl) = one["image"], one["target"]
    assert brk.shape == full[0].shape and brk.dtype == torch.uint8
    assert torch.equal(fu, full[0]) and int((brk & fl).sum()) == 0 and torch.equal(brk | fl, fu)
    assert np.array_equal(fl.cpu().numpy(), K.cut(full[:1].cpu().numpy(), rc.last.cpu().numpy())[2][0])


def _batch(b, size, seed):
    from ctunet_b200.synthetic import make_training_batch
    from ctunet_b200.utilities import pack_mask_bits
    img, (sk_t, _) = make_training_batch(b, 2, size, seed=seed, device=DEV)
    full = sk_t[:, 1].to(torch.uint8).contiguous()
    return full, pack_mask_bits(full), img[0, 1].contiguous()


def _net():
    import ctunet_b200 as C
    C.set_compute_dtype("bf16")
    torch.manual_seed(0)
    return C.UNetSP().to(DEV).train()


def test_no_host_synchronisation():
    from ctunet_b200 import RandomAffine, RandomCraniectomy
    from ctunet_b200.trainer import TrainStep
    full, bits, atlas = _batch(2, 32, 8)
    rc = RandomCraniectomy()
    rc({"image": full})                                                   # library load, first-draw state
    step = TrainStep(_net(), "double", lr=1e-5, graph=True, craniectomy=RandomCraniectomy(), augment=RandomAffine())
    for _ in range(3):                                                    # eager warm-up (plans, allocator) and the capture
        step.step_from_skull_bits(bits, (32, 32, 32), atlas)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        rc({"image": full})
        rc.draw(bits, (32, 32, 32))
        for _ in range(2):
            step.step_from_skull_bits(bits, (32, 32, 32), atlas)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("fmt", ["bits", "u8"])
@pytest.mark.parametrize("augment", [False, True])
def test_skull_step_equals_plain_step_on_oracle_masks(graph, fmt, augment):
    """TrainStep(craniectomy=...).step_from_skull_bits / step_from_skulls against a plain TrainStep.step_from_bits fed the
    oracle's masks for the holes (and transforms) the step drew, two identically initialised UNetSP: the step inputs bit
    for bit; loss components and parameters within the tolerances of the eager-versus-graph step tests (the training
    step itself is not bitwise reproducible from run to run)."""
    from ctunet_b200 import RandomAffine, RandomCraniectomy
    from ctunet_b200.trainer import TrainStep
    from ctunet_b200.utilities import encode_flaprec_bits, pack_mask_bits
    full, bits, atlas = _batch(2, 32, 4)
    vol = tuple(full.shape[1:])
    net_c, net_p = _net(), _net()
    torch.manual_seed(7)
    cs = TrainStep(net_c, "double", lr=1e-5, graph=graph, craniectomy=RandomCraniectomy(),
                   augment=RandomAffine(rotate=20, translate=4) if augment else None)
    plain = TrainStep(net_p, "double", lr=1e-5, graph=graph)
    host = full.cpu().numpy()
    drawn = []
    for _ in range(4):
        ca = (cs.step_from_skull_bits(bits, vol, atlas) if fmt == "bits" else cs.step_from_skulls(full, atlas)).tolist()
        hole = cs.last_craniectomy()
        drawn.append(hole.clone())
        mats = cs.last_affine()[1] if augment else None
        ref = [torch.from_numpy(m).to(DEV) for m in K.encode(host, hole.cpu().numpy(), None if mats is None else mats.cpu().numpy())]
        cp = plain.step_from_bits(*[pack_mask_bits(m) for m in ref], vol, atlas).tolist()
        assert ca == pytest.approx(cp, rel=2e-2, abs=2e-2)
        ref_img, _ = encode_flaprec_bits(*[pack_mask_bits(m) for m in ref], vol, atlas)
        image, fm, lm = _encode(1 if fmt == "bits" else 0, bits if fmt == "bits" else full, hole, mats, atlas, vol)
        assert torch.equal(image, ref_img) and torch.equal(fm, ref[1]) and torch.equal(lm, ref[2])
        if graph and cs._graph is not None:
            assert all(torch.equal(a, b) for a, b in zip(cs._static, plain._static))
    assert all(not torch.equal(drawn[i], drawn[i + 1]) for i in range(3))
    if graph:
        assert cs.launches_per_step == plain.launches_per_step
    sa, sp = net_c.state_dict(), net_p.state_dict()
    for k in sa:
        if k.endswith("num_batches_tracked"):
            assert int(sa[k]) == int(sp[k]), k
        elif "running" in k:
            assert torch.allclose(sa[k], sp[k], rtol=5e-2, atol=2e-2 * float(sa[k].abs().max()) + 1e-6), k
        elif not k.startswith("cblock"):
            assert float((sa[k] - sp[k]).abs().max()) <= 1e-4, k


def test_graph_and_eager_steps_draw_the_same_holes():
    from ctunet_b200 import RandomCraniectomy
    from ctunet_b200.trainer import TrainStep
    full, bits, atlas = _batch(2, 32, 5)
    hist = []
    for graph in (False, True):
        torch.manual_seed(11)
        step = TrainStep(_net(), "double", lr=1e-5, graph=graph, craniectomy=RandomCraniectomy(0.8))
        ps, cs = [], []
        for _ in range(5):                                # 2 eager warm-up steps, the capture, 2 replays
            cs.append(step.step_from_skull_bits(bits, (32, 32, 32), atlas).tolist())
            ps.append(step.last_craniectomy().clone())
        hist.append((ps, cs))
        if graph:
            assert step._graph is not None
    (pe, ce), (pg, cg) = hist
    assert all(torch.equal(a, b) for a, b in zip(pe, pg))
    assert all(not torch.equal(pg[i], pg[i + 1]) for i in range(4))    # fresh holes on every replay
    for a, b in zip(ce, cg):
        assert a == pytest.approx(b, rel=2e-2, abs=2e-2)


def test_errors_before_any_launch(monkeypatch):
    from ctunet_b200 import RandomCraniectomy, _lib
    from ctunet_b200 import trainer as T
    from ctunet_b200.trainer import TrainStep
    from ctunet_b200 import utilities as U
    full, bits, atlas = _batch(2, 32, 6)
    vol = (32, 32, 32)
    step = TrainStep(_net(), "double", lr=1e-5, craniectomy=RandomCraniectomy())
    plain = TrainStep(_net(), "double", lr=1e-5)
    img = torch.zeros((2, 2) + vol, device=DEV)
    n0 = _lib.launches
    with pytest.raises(ValueError):
        step(img, (full, full))                                          # masks already cut
    with pytest.raises(ValueError):
        step.step_from_masks(full, full, full, atlas)
    with pytest.raises(ValueError):
        step.step_from_bits(bits, bits, bits, vol, atlas)
    with pytest.raises(ValueError):
        plain.step_from_skulls(full, atlas)                              # no craniectomy
    with pytest.raises(ValueError):
        plain.step_from_skull_bits(bits, vol, atlas)
    with pytest.raises(TypeError):
        step.step_from_skulls(full.float(), atlas)
    with pytest.raises(RuntimeError):
        step.step_from_skulls(full.cpu(), atlas)
    with pytest.raises(ValueError):
        step.step_from_skull_bits(bits, (32, 32, 16), atlas)
    with pytest.raises(TypeError):
        step.step_from_skull_bits(bits, vol, atlas.double())
    with pytest.raises(TypeError):
        TrainStep(_net(), "double", craniectomy=object())
    with pytest.raises(TypeError):
        RandomCraniectomy().draw(full.float())
    monkeypatch.setattr(U, "radius_bounds", lambda shape: (5, 5))
    with pytest.raises(ValueError):
        step.step_from_skulls(full, atlas)                               # empty radius range
    monkeypatch.undo()
    monkeypatch.setattr(T, "FUSED_HEAD_LOSS", False)
    with pytest.raises(ValueError):
        step.step_from_skulls(full, atlas)
    assert _lib.launches == n0
    assert step.last_craniectomy() is None
