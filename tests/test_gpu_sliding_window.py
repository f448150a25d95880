"""GPU: overlapping sliding-window inference (preprocess.sliding_window_predict, DESIGN.md section 7b) against the CPU
oracle of tests/window_oracle.py, against the non-overlapping sliding_window_argmax, the determinism of the integer
accumulators, the any-window patch gather and the argument checks."""
import pytest
import torch
import torch.nn.functional as F

import window_oracle as W

pytestmark = pytest.mark.gpu

DEV = "cuda"
TOL = {"fp32": 1e-4, "bf16": 2e-2}
_ORACLE = {}


def _net(name, mode):
    import ctunet_b200 as C
    C.set_compute_dtype(mode)
    torch.manual_seed(0)
    net = getattr(C, name)().to(DEV).eval()
    C.set_compute_dtype("bf16")
    return net


def _vol(cin, shape, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand((cin,) + tuple(shape), generator=g) > 0.7).float()


def _oracle(name, shape, patch, overlap, blend, seed):
    key = (name, shape, patch, overlap, blend, seed)
    if key not in _ORACLE:
        from oracle import unet_oracle as O
        cfg = O.PRESETS[name]
        sd = O.build_state_dict(cfg, seed=0)
        vol = _vol(cfg.input_channels, shape, seed)
        _ORACLE[key] = (vol,) + W.predict(sd, cfg, vol, patch, overlap, blend)[:2]
    return _ORACLE[key]


def _check(name, mode, shape, patch, overlap, blend, seed=3, batch=4):
    from ctunet_b200 import preprocess as P
    vol, ref, ref_lab = _oracle(name, shape, patch, overlap, blend, seed)
    net = _net(name, mode)
    labels, probs = P.sliding_window_predict(net, vol.to(DEV), patch=patch, overlap=overlap, blend=blend, batch=batch,
                                             probs=True)
    assert not net.training
    assert len(labels) == len(probs) == len(ref)
    tol = TOL[mode]
    for lab, pr, r, rl in zip(labels, probs, ref, ref_lab):
        assert lab.shape == tuple(shape) and lab.dtype == torch.float32
        assert pr.shape == r.shape and pr.dtype == torch.float32
        scale = float(r.abs().max())
        err = float((pr.cpu().double() - r).abs().max()) / scale
        assert err < tol, (name, mode, blend, err)
        band = W.margin(r) <= tol * scale                     # labels may differ only inside the tie band
        mism = lab.cpu() != rl
        assert not bool((mism & ~band).any()), (name, mode, blend, int((mism & ~band).sum()))
        print("%s %s %s: max rel err %.2e, %d voxels in the tie band, %d of them differ"
              % (name, mode, blend, err, int(band.sum()), int(mism.sum())))


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("blend", ["constant", "gaussian"])
@pytest.mark.parametrize("name", ["UNet", "UNetSP", "UNetSPSmall", "recAE_v2_fixed"])
def test_matches_oracle_any_shape(name, blend, mode):
    """Depth 24 < patch 32, width 70 (not a multiple of 4), x origins 0, 16, 32, 38; every head kind."""
    _check(name, mode, (24, 56, 70), 32, 0.5, blend)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_matches_oracle_at_the_trained_patch_size(mode):
    """128^3 windows on [2, 160, 200, 136] at overlap 0.25: a 2 x 2 x 2 grid."""
    _check("UNetSP", mode, (160, 200, 136), 128, 0.25, "gaussian")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["UNetSP", "recAE_v2_fixed"])
def test_overlap_zero_equals_sliding_window_argmax(name, mode):
    """Overlap 0 with constant weights covers every voxel once with weight 1: v * 2^40 is an exact integer for every
    v >= 2^-16, so the labels are sliding_window_argmax's wherever the larger channel is at least that."""
    from ctunet_b200 import preprocess as P
    net = _net(name, mode)
    cin = 2 if name == "UNetSP" else 1
    vol = _vol(cin, (64, 64, 96), 5).to(DEV)
    want = P.sliding_window_argmax(net, vol, patch=32, batch=4)
    labels, probs = P.sliding_window_predict(net, vol, patch=32, overlap=0.0, blend="constant", batch=4, probs=True)
    for a, b, p in zip(labels, want, probs):
        ok = p.max(0).values >= 2.0 ** -16
        assert bool(ok.all()) or int((~ok).sum()) < ok.numel() // 1000
        assert torch.equal(a[ok], b[ok])


def test_accumulators_are_deterministic():
    """Bit-identical int64 sums: graph replay against eager, batch 1 against batch 4, a permuted window order, and the
    two shards of a 2-rank split summed in one process against the single-rank pass."""
    from ctunet_b200 import preprocess as P
    net = _net("UNetSP", "bf16")
    vol = _vol(2, (24, 56, 70), 9).to(DEV)
    args = dict(patch=32, overlap=0.5, blend="gaussian", sigma_scale=0.125)

    def acc(batch, graph, rank=0, world=1):
        a, axes = P._accumulate_windows(net, vol, args["patch"], args["overlap"], args["blend"], args["sigma_scale"],
                                        batch, graph, rank, world)
        return a.clone(), axes

    ref, axes = acc(4, True)
    assert ref.dtype == torch.int64 and ref.shape == (4, 24, 56, 70)
    assert bool((ref[0] + ref[1] > 0).all())                          # every voxel is covered
    assert torch.equal(acc(4, False)[0], ref)
    assert torch.equal(acc(1, True)[0], ref)
    assert torch.equal(acc(3, True)[0], ref)                           # 12 windows: ragged-free; 5 would leave a tail
    assert torch.equal(acc(5, True)[0], ref)
    assert torch.equal(acc(4, True, 0, 2)[0] + acc(4, True, 1, 2)[0], ref)
    wins = [(z, y, x) for z in axes[0] for y in axes[1] for x in axes[2]]
    perm = torch.randperm(len(wins), generator=torch.Generator().manual_seed(1)).tolist()
    org = torch.tensor([wins[i] for i in perm], dtype=torch.int32, device=DEV)
    wt = torch.tensor(P.window_weights(32, "gaussian"), dtype=torch.float32).expand(3, 32).contiguous().to(DEV)
    a = torch.zeros_like(ref)
    for i in range(0, len(wins), 4):
        net.accumulate_windows(vol=vol, origins=org[i:i + 4], patch=32, weights=wt, acc=a)
    assert torch.equal(a, ref)
    # the public entry point: graph and eager give the same labels and blended values bit for bit
    l1, p1 = P.sliding_window_predict(net, vol, batch=4, probs=True, **args)
    l2, p2 = P.sliding_window_predict(net, vol, batch=4, probs=True, graph=False, **args)
    for u, v in zip(l1 + p1, l2 + p2):
        assert torch.equal(u, v)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_patch_gather_any_window(mode):
    """ctu_pack_patches with windows crossing every face of the volume (and an odd width) against slicing a zero-padded
    volume; the float4 path (width and x origin multiples of 4, window inside) against the same reference."""
    from ctunet_b200.engine import Engine
    p = 8
    for (c, d, h, w) in ((3, 12, 13, 15), (9, 16, 16, 24)):
        vol = torch.randn(c, d, h, w, device=DEV)
        org = [(-3, 0, 0), (0, -5, 4), (0, 0, -2), (d - 5, 0, 0), (0, h - 3, 0), (0, 0, w - 6), (-8, -8, -8), (d, h, w),
               (2, 3, 4), (1, 2, 8), (-1, h - 7, w - 1)]
        o = torch.tensor(org, dtype=torch.int32, device=DEV)
        eng = Engine(torch.device(DEV), mode, record=False)
        eng.patch_src = (vol, o, p)
        a = eng.pack(None)
        got = eng.unpack(a)                                          # fp32 [B, C, p, p, p]
        pad = F.pad(vol, (p, p, p, p, p, p))
        want = torch.stack([pad[:, z + p:z + 2 * p, y + p:y + 2 * p, x + p:x + 2 * p] for z, y, x in org])
        if mode == "bf16":
            want = want.to(torch.bfloat16).float()
        assert torch.equal(got, want), (c, d, h, w)


def test_invalid_arguments_raise():
    import ctunet_b200 as C
    from ctunet_b200 import preprocess as P
    net = _net("UNetSP", "bf16")
    vol = _vol(2, (24, 56, 70), 1).to(DEV)
    with pytest.raises(RuntimeError):
        P.sliding_window_predict(net, vol.cpu(), patch=32)
    for kw in (dict(overlap=1.0), dict(overlap=-0.1), dict(blend="cosine"), dict(sigma_scale=0.0), dict(patch=24),
               dict(patch=12)):
        with pytest.raises(ValueError):
            P.sliding_window_predict(net, vol, **dict(dict(patch=32), **kw))
    with pytest.raises(ValueError):
        P.sliding_window_predict(net, vol[:1].contiguous(), patch=32)          # Cin does not match the model
    with pytest.raises(TypeError):
        P.sliding_window_predict(net, vol.double(), patch=32)
    with pytest.raises(ValueError):
        P.sliding_window_predict(net, vol[0], patch=32)
    plain = C.UNet(apply_sigmoid=False).to(DEV)                                 # unbounded head: no fixed-point sums
    with pytest.raises(RuntimeError):
        P.sliding_window_predict(plain, vol[:1].contiguous(), patch=32)
    assert plain.training                                                       # the mode is restored on error too


def test_full_size_volume_overlap_half():
    """A 224 x 512 x 512 volume (a shape sliding_window_argmax refuses at the 128^3 patch) at overlap 0.5: 147 windows."""
    from ctunet_b200 import preprocess as P
    net = _net("UNetSP", "bf16")
    vol = _vol(2, (224, 512, 512), 2).to(DEV)
    with pytest.raises(ValueError):
        P.sliding_window_argmax(net, vol, patch=128)
    labels = P.sliding_window_predict(net, vol, patch=128, overlap=0.5, batch=4)
    assert len(labels) == 2 and labels[0].shape == (224, 512, 512)
    assert bool(((labels[0] == 0) | (labels[0] == 1)).all()) and bool(((labels[1] == 0) | (labels[1] == 1)).all())
