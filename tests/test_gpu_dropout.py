"""Dropout3d (dropout_p > 0) on the fused path (GPU): the keep-factor kernels of csrc/dropout.cu, the BatchNorm+ReLU(+MaxPool)
kernels with keep factors against plain torch, and training / inference of the model classes against the CPU oracle fed
the masks the product drew (``net.dropout_keep()``)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import dropout_oracle as DO

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _eng(mode, record=True):
    from ctunet_b200.engine import Engine
    return Engine(torch.device(DEV), mode, record)


def _rnd(mode, t):
    return t if mode == "fp32" else t.to(torch.bfloat16).to(torch.float32)


def _close(a, b, mode, what=""):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    ref = max(b.abs().max().item(), 1e-6)
    err = (a - b).abs().max().item()
    lim = (1e-4 if mode == "fp32" else 1.2e-2) * ref
    assert err <= lim, "%s: max abs err %.3e > %.3e (ref max %.3e)" % (what, err, lim, ref)


def _kept(p):
    return float(np.float32(1) / (np.float32(1) - np.float32(p)))


def _keep_call(sites, n, seed, counter):
    """ctu_dropout3d_keep for [(site, channels, p)] -> list of [n, cpad] CPU tensors."""
    from ctunet_b200 import _lib
    cpads = [(c + 7) // 8 * 8 for _, c, _ in sites]
    buf = torch.full((n * sum(cpads),), -1.0, device=DEV)
    _lib.call("ctu_dropout3d_keep", len(sites), _lib.int_array([s[0] for s in sites]), _lib.int_array([s[1] for s in sites]),
              (_lib.c_float * len(sites))(*[s[2] for s in sites]), n, seed,
              counter.data_ptr() if counter is not None else None, buf.data_ptr(), _lib.stream_ptr())
    out, off = [], 0
    for cp in cpads:
        out.append(buf[off:off + n * cp].view(n, cp).cpu())
        off += n * cp
    return out


# ---------------------------------------------------------------------------------------------------- keep factors
def test_keep_factor_statistics_and_values():
    n, c = 512, 253
    counter = torch.zeros(1, dtype=torch.int64, device=DEV)
    sites = [(0, c, 0.1), (3, c, 0.5), (5, 13, 1.0), (6, 9, 0.0)]
    k01, k05, k1, k0 = _keep_call(sites, n, 0x1234_5678_9ABC, counter)
    assert int(counter) == 1
    for k, p in ((k01, 0.1), (k05, 0.5)):
        real = k[:, :c]
        assert torch.equal(k[:, c:], torch.zeros(n, k.shape[1] - c))                    # pad lanes
        vals = set(real.unique().tolist())
        assert vals == {0.0, _kept(p)}, vals                                               # exactly 0 or 1/(1-p) in fp32
        kept = int((real != 0).sum())
        tot = real.numel()
        sigma = (tot * p * (1 - p)) ** 0.5
        assert abs(kept - tot * (1 - p)) <= 5 * sigma, (p, kept, tot)
    assert float(k1.abs().sum()) == 0.0                                                    # p = 1: everything dropped
    assert torch.equal(k0[:, :9], torch.ones(n, 9)) and float(k0[:, 9:].abs().sum()) == 0.0
    # the next pass draws a different mask; the same (seed, pass) reproduces it
    k01b = _keep_call(sites[:1], n, 0x1234_5678_9ABC, counter)[0]
    assert int(counter) == 2 and not torch.equal(k01b, k01)
    again = _keep_call(sites[:1], n, 0x1234_5678_9ABC, torch.zeros(1, dtype=torch.int64, device=DEV))[0]
    assert torch.equal(again, k01)
    assert torch.equal(_keep_call(sites[:1], n, 0x1234_5678_9ABC, None)[0], k01)            # no counter: pass 0
    other_site = _keep_call([(1, c, 0.1)], n, 0x1234_5678_9ABC, None)[0]
    assert not torch.equal(other_site, k01)


# ---------------------------------------------------------------------------------------------------- BatchNorm kernels
def _keep_tensor(n, c, p, seed):
    g = torch.Generator().manual_seed(seed)
    cpad = (c + 7) // 8 * 8
    k = torch.zeros(n, cpad)
    k[:, :c] = (torch.rand(n, c, generator=g) >= p).float() * _kept(p)
    k[:, 0] = 0.0                      # a channel dropped in every sample
    if c > 1:
        k[:, 1] = _kept(p)             # and one kept everywhere
    return k


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("fold", [True, False])
@pytest.mark.parametrize("pool", [False, True])
@pytest.mark.parametrize("shape", [(2, 7, 4, 4, 8), (1, 14, 8, 6, 4), (3, 9, 2, 2, 2), (2, 5, 3, 5, 3)])
def test_bn_relu_drop_fwd_bwd(mode, fold, pool, shape, monkeypatch):
    """ctu_bn_relu_*_drop against F.batch_norm -> relu -> * k (-> max_pool3d): plain (odd dims: one voxel per thread; even:
    the 8-children structure), pooled, folded and separate finalisation (either side of BN_FOLD_MAX_VOXELS)."""
    from ctunet_b200 import engine as E
    n, c, d, h, w = shape
    if pool and (d % 2 or h % 2 or w % 2):
        pytest.skip("MaxPool3d(2) needs even dims")
    monkeypatch.setattr(E, "BN_FOLD_MAX_VOXELS", 1 << 40 if fold else 0)
    g = torch.Generator().manual_seed(3)
    x = _rnd(mode, torch.randn(*shape, generator=g) * 1.5 + 0.3)
    keep = _keep_tensor(n, c, 0.3, 5)
    bn_ref = torch.nn.BatchNorm3d(c)
    with torch.no_grad():
        bn_ref.weight.copy_(torch.rand(c, generator=g) + 0.5)
        bn_ref.bias.copy_(torch.randn(c, generator=g) * 0.2)
    bn_gpu = torch.nn.BatchNorm3d(c)
    bn_gpu.load_state_dict(bn_ref.state_dict())
    bn_gpu.to(DEV)
    xr = x.clone().requires_grad_()
    ar = F.relu(bn_ref(xr)) * keep[:, :c, None, None, None]
    outs_r = [ar] + ([F.max_pool3d(ar, 2, 2)] if pool else [])
    gr = [_rnd(mode, torch.randn(o.shape, generator=g)) for o in outs_r]
    torch.autograd.backward(outs_r, gr)

    eng = _eng(mode)
    y = eng.pack(x.to(DEV))
    res = eng.bn_relu(y, bn_gpu, True, extra_updates=0, pool=pool, keep=keep.to(DEV))
    res = res if pool else (res,)
    ss = res[0].bn["ss"].clone()            # the fp32 scale / shift / mean / invstd the kernels use
    for o, r, nm in zip(res, outs_r, ["a", "pooled"]):
        _close(eng.unpack(o), r, mode, what=nm)
    # batch statistics are those of y (BatchNorm precedes the dropout)
    assert torch.allclose(bn_gpu.running_mean.cpu(), bn_ref.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(bn_gpu.running_var.cpu(), bn_ref.running_var, rtol=1e-4, atol=1e-5)
    for o, gg in zip(res, gr):
        eng.agrads[id(o)] = eng.pack(gg.to(DEV))
    eng.run_tape()
    dyo = eng.unpack(eng.agrads[id(y)]).cpu()
    assert float(dyo[:, 0].abs().max()) == 0.0                         # the dropped channel passes no gradient
    if mode == "bf16" and pool:
        # routing exact except at windows within fp32 rounding of a flip (see tests/test_gpu_ops.py)
        import norm_head_oracle as NO
        cpad = (c + 7) // 8 * 8
        ss4 = tuple(ss.double().view(4, cpad)[:, :c].cpu())
        ref, err, gate, tie = NO.dy_error_with_ties(x, ss4, gr[0], gr[1], keep[:, :c], dyo)
        print("tie-marked: %d gates, %d windows" % (int(gate.sum()), int(tie.sum())))
        assert float(err.max()) <= 1.2e-2 * float(ref["dy"].abs().max()), "dy: max abs err %.3e" % float(err.max())
    else:
        _close(dyo, xr.grad, mode, what="dy")
    _close(eng.pgrads[id(bn_gpu.weight)], bn_ref.weight.grad, mode, what="dgamma")
    _close(eng.pgrads[id(bn_gpu.bias)], bn_ref.bias.grad, mode, what="dbeta")
    assert float(eng.pgrads[id(bn_gpu.weight)][0].abs()) == 0.0 and float(eng.pgrads[id(bn_gpu.bias)][0].abs()) == 0.0


def test_phase_major_input_refuses_keep_factors():
    from ctunet_b200 import _lib
    a = torch.zeros(1, 8, 2, 2, 2, 8, device=DEV)
    ss = torch.zeros(32, device=DEV)
    k = torch.ones(1, 8, device=DEV)
    with pytest.raises(RuntimeError, match="phase-major"):
        _lib.call("ctu_bn_relu_fwd_drop", _lib.CTU_F32, a.data_ptr(), ss.data_ptr(), a.data_ptr(), None, 8, 1, 4, 4, 4, 1,
                  k.data_ptr(), _lib.stream_ptr())


# ---------------------------------------------------------------------------------------------------- models
def _net(name, mode, p, seed=0):
    import ctunet_b200 as C
    C.set_compute_dtype(mode)
    torch.manual_seed(seed)
    net = getattr(C, name)()
    C.set_compute_dtype("bf16")
    for _, m, _ in net._dropout_sites():
        m.p = p
    return net.to(DEV)


def _data(name, size, batch, seed=7):
    from oracle import unet_oracle as O
    cfg = O.PRESETS[name]
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(batch, cfg.input_channels, size, size, size, generator=g)           # continuous: no pooling ties
    sk = (torch.rand(batch, size, size, size, generator=g) > 0.6).long()
    fl = ((torch.rand(batch, size, size, size, generator=g) > 0.8) & (sk > 0)).long()
    oh = lambda t: F.one_hot(t, 2).permute(0, 4, 1, 2, 3).float().contiguous()
    return cfg, x, oh(sk), oh(fl)


def _loss(cfg, out, sk, fl):
    from oracle import unet_oracle as O
    if cfg.head == "plain":
        return O.loss_single_output(out, sk, 1.0, 1.0)
    return O.loss_double_output(out, (sk, fl), 1.0, 1.0)


def _oracle(cfg, sd0, x, keep, sk, fl, act_round=None):
    from oracle import unet_oracle as O
    sd = {k: v.detach().cpu().clone() for k, v in sd0.items()}
    pn = [k for k in sd if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))]
    for k in pn:
        sd[k].requires_grad_()
    out = DO.unet_forward(sd, x.clone().requires_grad_(), cfg, training=True, act_round=act_round,
                         dropout_keep={k: v.cpu() for k, v in keep.items()})
    loss, comps = _loss(cfg, out, sk, fl)
    loss.backward()
    return sd, pn, out, comps


def _step(net, cfg, x, sk, fl):
    out = net(x.to(DEV).requires_grad_())
    loss, comps = _loss(cfg, out, sk.to(DEV), fl.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    return out, comps


@pytest.mark.parametrize("name,mode,size", [("UNetSP", "fp32", 32), ("UNetSPSmall", "fp32", 32), ("recAE_v2_fixed", "fp32", 32),
                                            ("UNet4_2IC", "fp32", 32), ("UNetSP", "bf16", 32), ("recAE_v2_fixed", "bf16", 32),
                                            ("UNetSP", "fp32", 128)])
def test_train_step_with_dropout_matches_oracle(name, mode, size):
    cfg, x, sk, fl = _data(name, size, 2)
    net = _net(name, mode, 0.3).train()
    sd0 = {k: v.detach().clone() for k, v in net.state_dict().items()}
    out, comps = _step(net, cfg, x, sk, fl)
    keep = net.dropout_keep()
    sites = [nm for nm, m, _ in net._dropout_sites()]
    assert sorted(keep) == sorted(sites)
    assert any(float((k == 0).float().mean()) > 0 for k in keep.values())
    sd, pn, ref, rcomps = _oracle(cfg, sd0, x, keep, sk, fl)
    outs = out if isinstance(out, tuple) else (out,)
    refs = ref if isinstance(ref, tuple) else (ref,)
    named = dict(net.named_parameters())
    if mode == "fp32":
        for o, r in zip(outs, refs):
            _close(o, r, "fp32", what="output")
        for k, v in rcomps.items():
            assert float(comps[k].detach()) == pytest.approx(float(v.detach()), rel=1e-4, abs=1e-6), k
        for k in pn:
            if sd[k].grad is None:                # the generic UNet's discarded center block
                assert named[k].grad is None, k
                continue
            gr, gg = sd[k].grad.double(), named[k].grad.cpu().double()
            if float(gr.norm()) < 1e-5:           # conv biases ahead of BatchNorm: analytically zero gradient
                assert float(gg.norm()) < 1e-4, k
                continue
            rel = float((gg - gr).norm() / gr.norm())
            assert rel < 1e-2, "%s: normwise gradient error %.2e" % (k, rel)
    else:
        for o, r in zip(outs, refs):
            err = float((o.detach().cpu() - r.detach()).abs().max() / r.detach().abs().max())
            assert err < 2e-2, err
        for k, v in rcomps.items():
            assert abs(float(comps[k].detach()) - float(v.detach())) < 5e-3, k
        dot = nr = ng = 0.0
        worst = 1.0
        for k in pn:
            if sd[k].grad is None:
                assert named[k].grad is None, k
                continue
            gr, gg = sd[k].grad.double(), named[k].grad.cpu().double()
            if float(gr.norm()) < 1e-5:
                continue
            worst = min(worst, float((gg * gr).sum() / (gg.norm() * gr.norm())))
            dot += float((gg * gr).sum())
            nr += float(gr.norm() ** 2)
            ng += float(gg.norm() ** 2)
        assert worst > 0.7 and dot / (nr * ng) ** 0.5 > 0.95, (worst, dot / (nr * ng) ** 0.5)
    # BatchNorm buffers: the forward update and the checkpoint's second one at backward time
    sdn = net.state_dict()
    for k in sd:
        if k.endswith("num_batches_tracked"):
            assert int(sdn[k]) == int(sd[k]), k
        elif k.endswith(("running_mean", "running_var")):
            assert torch.allclose(sdn[k].cpu(), sd[k], rtol=1e-3 if mode == "bf16" else 1e-4,
                                  atol=1e-3 if mode == "bf16" else 1e-6), k


def test_masks_reproducible_and_counted_inside_the_captured_step():
    """Same torch.manual_seed -> same masks; a TrainStep(graph=True) run draws exactly the masks of the eager steps counted
    from the same start (warm-up steps included): the pass counter advances inside the graph."""
    from ctunet_b200.trainer import TrainStep
    cfg, x, sk, fl = _data("UNetSP", 16, 2)
    xg, tg = x.to(DEV), (sk.to(DEV), fl.to(DEV))
    runs = []
    for graph in (False, True):
        net = _net("UNetSP", "bf16", 0.3, seed=11)
        torch.manual_seed(1234)
        step = TrainStep(net, "double", graph=graph)
        masks = []
        for _ in range(4):
            step(xg, tg)
            torch.cuda.synchronize()
            masks.append({k: v.clone() for k, v in net.dropout_keep().items()})
        runs.append(masks)
    for a, b in zip(*runs):
        assert a.keys() == b.keys()
        for k in a:
            assert torch.equal(a[k], b[k]), k
    m = runs[1]
    assert any(not torch.equal(m[2][k], m[3][k]) for k in m[2])          # two replays: fresh masks


def test_dropout_training_reduces_loss_in_graph_mode():
    from ctunet_b200.trainer import TrainStep
    cfg, x, sk, fl = _data("UNetSP", 64, 2)
    net = _net("UNetSP", "bf16", 0.1)
    step = TrainStep(net, "double", lr=1e-3, graph=True)
    xg, tg = x.to(DEV), (sk.to(DEV), fl.to(DEV))
    losses = [float(step(xg, tg)[-1]) for _ in range(20)]
    assert step.launches_per_step is not None
    assert np.isfinite(losses).all()
    assert np.mean(losses[-3:]) < np.mean(losses[:3]), losses
    with pytest.raises(RuntimeError, match="Dropout3d"):
        net.d_blocks[0].block[6].p = 0.2
        step(xg, tg)


def test_monte_carlo_inference_matches_eval_oracle():
    from oracle import unet_oracle as O
    cfg, x, _, _ = _data("recAE_v2_fixed", 32, 2)
    net = _net("recAE_v2_fixed", "fp32", 0.4)
    with torch.no_grad():           # non-trivial running statistics
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm3d):
                m.running_mean.uniform_(-0.1, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    net.eval()
    for _, m, _ in net._dropout_sites():
        m.train()
    with torch.no_grad():
        out1 = net(x.to(DEV))
        keep1 = {k: v.clone() for k, v in net.dropout_keep().items()}
        out2 = net(x.to(DEV))
    torch.cuda.synchronize()
    assert not torch.equal(out1, out2)
    sd = {k: v.cpu() for k, v in net.state_dict().items()}
    ref = DO.unet_forward(sd, x, cfg, training=False, dropout_keep={k: v.cpu() for k, v in keep1.items()})
    _close(out1, ref, "fp32", what="MC-dropout output")
    # every module in eval mode: deterministic, the plain eval forward
    net.eval()
    with torch.no_grad():
        a, b = net(x.to(DEV)), net(x.to(DEV))
    assert torch.equal(a, b)
    _close(a, DO.unet_forward(sd, x, cfg, training=False), "fp32", what="eval output")


def test_dropin_graph_replays_draw_fresh_masks(monkeypatch):
    from ctunet_b200 import models as M
    monkeypatch.setattr(M, "DROPIN_GRAPH", True)
    cfg, x, sk, fl = _data("UNetSP", 16, 2)
    net = _net("UNetSP", "bf16", 0.3).train()
    masks = []
    for _ in range(5):
        _step(net, cfg, x, sk, fl)
        masks.append({k: v.clone() for k, v in net.dropout_keep().items()})
        net.zero_grad(set_to_none=True)
    st = next(iter(net._dropin_graphs.values()))
    assert st.fwd is not None and st.bwd is not None                 # calls 3.. replayed captured graphs
    for i in (2, 3):
        assert any(not torch.equal(masks[i][k], masks[i + 1][k]) for k in masks[i])


def test_data_parallel_replica_trains_with_dropout():
    from torch.nn.parallel import replicate
    cfg, x, sk, fl = _data("UNetSP", 16, 2)
    net = _net("UNetSP", "fp32", 0.3).train()
    rep = replicate(net, [torch.cuda.current_device()])[0]
    assert getattr(rep, "_is_replica", False)
    sd0 = {k: v.detach().clone() for k, v in net.state_dict().items()}
    out, comps = _step(rep, cfg, x, sk, fl)
    keep = net.dropout_keep()                  # the replica shares the model's random state
    assert len(keep) == 8
    _, _, ref, rcomps = _oracle(cfg, sd0, x, keep, sk, fl)
    for o, r in zip(out, ref):
        _close(o, r, "fp32", what="replica output")
    assert all(p.grad is not None for p in net.parameters() if p.requires_grad and p.dim() > 1)


def test_inactive_dropout_is_bit_identical_and_launches_nothing():
    """dropout_p = 0 and Dropout3d modules in eval mode inside a training net: the same launches and bit-identical results
    as a net built without dropout."""
    from ctunet_b200.trainer import TrainStep
    cfg, x, sk, fl = _data("UNetSP", 16, 2)
    xg, tg = x.to(DEV), (sk.to(DEV), fl.to(DEV))
    res = []
    for variant in ("none", "eval"):
        net = _net("UNetSP", "bf16", 0.0 if variant == "none" else 0.5)
        if variant == "eval":
            net.train()
            for _, m, _ in net._dropout_sites():
                m.eval()
            out = net(xg.clone().requires_grad_())
        else:
            out = net.train()(xg.clone().requires_grad_())
        torch.cuda.synchronize()
        assert net.dropout_keep() == {}
        res.append(out)
    for a, b in zip(*res):
        assert torch.equal(a, b)
    launches = []
    for p in (0.0, 0.0):
        net = _net("UNetSP", "bf16", p)
        step = TrainStep(net, "double", graph=True)
        for _ in range(3):
            step(xg, tg)
        launches.append(step.launches_per_step)
    net = _net("UNetSP", "bf16", 0.2)
    step = TrainStep(net, "double", graph=True)
    for _ in range(3):
        step(xg, tg)
    assert launches[0] == launches[1]
    assert step.launches_per_step == launches[0] + 1            # the one mask launch (its kernels: no new launches)
