"""Parity AT THE BENCHMARKED CONFIGURATION (GPU): one bf16 training step of the networks on 64^3 / 128^3 volumes of the
bench's own synthetic skull phantom against the CPU oracle on the SAME tensors, plus the code paths only large tensors
take (un-folded training BatchNorm finalisation, d-chunked persistent convolution schedules, three fused up levels).

Tolerances (north_star): bf16 outputs within 2e-2 relative of the fp32 reference, every loss component (Dice, CE) within
5e-3 absolute.  Gradients: see test_bf16_gradients_sit_on_the_noise_floor_of_the_format.
"""
import types

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _relerr(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def _build(name, mode="bf16"):
    import ctunet_b200 as C
    C.set_compute_dtype(mode)
    torch.manual_seed(0)
    net = getattr(C, name)()
    C.set_compute_dtype("bf16")
    return net.to(DEV)


def _oracle_step(name, x, target, act_round=None):
    from oracle import unet_oracle as O
    cfg = O.PRESETS[name]
    sd = O.build_state_dict(cfg, seed=0)
    pn = [k for k in sd if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))]
    for k in pn:
        sd[k].requires_grad_()
    out = O.unet_forward(sd, x, cfg, training=True, act_round=act_round)
    if isinstance(out, tuple):
        loss, comps = O.loss_double_output(out, target, 1.0, 1.0)
    else:
        loss, comps = O.loss_single_output(out, target, 1.0, 1.0)
    loss.backward()
    return sd, pn, out, comps


def _product_step(name, x, target, mode="bf16"):
    import ctunet_b200 as C
    net = _build(name, mode).train()
    fake = types.SimpleNamespace(params=dict(dice_lambda=1.0, ce_lambda=1.0, save_dice_plots=False, save_hd_plots=False),
                                 losses_and_metrics={}, pt_loss=None)
    xg = x.to(DEV).requires_grad_()
    out = net(xg)
    if isinstance(out, tuple):
        C.FlapRecWithShapePriorDoubleOut.comp_losses_metrics(fake, out, tuple(t.to(DEV) for t in target), 0, 1, verbose=False)
    else:
        C.ProblemHandler.comp_losses_metrics(fake, out, target.to(DEV), 0, 1, verbose=False)
    fake.pt_loss.backward()
    torch.cuda.synchronize()
    return net, out, fake


@pytest.mark.parametrize("name,batch,size", [("UNetSP", 4, 64), ("UNetSP", 2, 128), ("recAE_v2_fixed", 2, 64),
                                             ("UNet4_2IC", 1, 64)])
def test_bf16_train_step_at_benchmark_sizes_matches_oracle(name, batch, size):
    """Forward outputs, every loss component, BatchNorm buffers (incl. the double update of the reentrant checkpoint and
    the once-updated dead center block) and the set of parameters that receive a gradient -- on the bench's phantom."""
    from oracle import unet_oracle as O
    cfg = O.PRESETS[name]
    x, (sk_t, fl_t) = O.make_training_batch(batch, cfg.input_channels, size, seed=1234)
    target = (sk_t, fl_t) if cfg.head != "plain" else sk_t
    sd, pn, ref_out, comps = _oracle_step(name, x, target)
    net, out, fake = _product_step(name, x, target)
    outs = out if isinstance(out, tuple) else (out,)
    refs = ref_out if isinstance(ref_out, tuple) else (ref_out,)
    for o, r in zip(outs, refs):
        assert o.shape == r.shape
        assert _relerr(o, r) < 2e-2
    for k, v in comps.items():
        assert abs(fake.losses_and_metrics[k][0] - float(v)) < 5e-3, (k, fake.losses_and_metrics[k][0], float(v))
    named = dict(net.named_parameters())
    assert [k for k in pn if sd[k].grad is None] == [k for k in pn if named[k].grad is None]
    got = net.state_dict()
    worst_mean = 0.0
    for k, v in sd.items():
        if k.endswith("num_batches_tracked"):
            assert int(got[k]) == int(v), k
        elif k.endswith("running_mean"):
            # the batch mean within 1 % of the channel's batch standard deviation (bf16 storage of the convolution output);
            # running_var = 0.9^u + (1 - 0.9^u) * unbiased batch variance after u updates
            u = int(sd[k.replace("running_mean", "num_batches_tracked")])
            w_old = 0.9 ** u
            std = ((sd[k.replace("running_mean", "running_var")] - w_old) / (1 - w_old)).clamp_min(0).sqrt()
            err = ((got[k].cpu() - v).abs() / ((1 - w_old) * std.clamp_min(1e-6))).max().item()
            worst_mean = max(worst_mean, err)
            assert err < 1e-2, (k, err)
        elif k.endswith("running_var"):
            assert torch.allclose(got[k].cpu(), v, rtol=3e-2, atol=1e-5), k
    print("%s %dx%d^3: worst batch-mean error = %.4f of the channel's batch std" % (name, batch, size, worst_mean))
    # whole-gradient direction against the fp32 reference (per-tensor accuracy is the subject of the next test)
    dot = nr = ng = 0.0
    for k in pn:
        if sd[k].grad is None or float(sd[k].grad.norm()) < 1e-6:
            continue
        gr, gg = sd[k].grad.double(), named[k].grad.cpu().double()
        dot, nr, ng = dot + float((gg * gr).sum()), nr + float(gr.norm() ** 2), ng + float(gg.norm() ** 2)
    assert dot / (nr * ng) ** 0.5 > 0.95


@pytest.mark.parametrize("name,batch,size", [("UNetSP", 2, 64), ("UNetSP", 1, 128)])
def test_bf16_gradients_sit_on_the_noise_floor_of_the_format(name, batch, size):
    """Per-tensor gradient accuracy of the bf16 product path at the benchmarked volume size, on continuous (tie-free) inputs,
    within ``step_oracle.noise_floor`` of the CPU oracle (bf16g' = the input perturbed by 3e-7 relative, i.e. one or two
    fp32 ulps).  Two equally valid bf16 evaluations of this network are tens of percent apart per deep tensor
    (profiles/r2_grad_parity_*.txt: the CPU oracle against itself); the bound is that distance."""
    from oracle import unet_oracle as O
    from step_oracle import noise_floor, rel_err
    cfg = O.PRESETS[name]
    g = torch.Generator().manual_seed(99)
    x = torch.rand(batch, cfg.input_channels, size, size, size, generator=g)
    xp = x * (1 + 3e-7 * torch.randn(x.shape, generator=g))
    _, target = O.make_training_batch(batch, cfg.input_channels, size, seed=77)
    bounds, comps_w = noise_floor(name, O.build_state_dict(cfg, seed=0), x, xp, target)
    net, out, fake = _product_step(name, x, target)
    named = dict(net.named_parameters())
    for k, v in comps_w.items():
        assert abs(fake.losses_and_metrics[k][0] - float(v)) < 1e-3, k
    worst_ratio, rows = 0.0, []
    num = den = 0.0
    for k, ent in bounds.items():
        if ent is None:
            assert named[k].grad is None, k
            continue
        ref, bound, ref_acc = ent
        if bound is None:                    # conv biases ahead of BatchNorm: analytically zero
            continue
        got = named[k].grad.cpu()
        err = rel_err(got, ref)
        rows.append((k, err, ref_acc))
        worst_ratio = max(worst_ratio, err / bound)
        assert err <= bound, "%s: error %.4f vs the bf16 oracle, bound %.4f, reference accumulation error %.4f" % (
            k, err, bound, ref_acc)
        num += float((got.double() - ref.double()).norm() ** 2)
        den += float(ref.double().norm() ** 2)
    whole = (num / den) ** 0.5
    print("%s %dx%d^3: whole-gradient error vs the bf16 oracle %.4f; worst tensor at %.2f of its bound" % (name, batch, size, whole,
                                                                                                  worst_ratio))
    assert whole < 0.03
    # the tensors that carry the gradient norm (the last blocks, the head) are tight in absolute terms
    for k, err, ref_acc in rows:
        if k.startswith(("last_conv", "u_blocks.3.block.5", "d_blocks.0.block.4")):
            assert err < 0.01 + ref_acc, (k, err)


def test_unfolded_training_batchnorm_matches_torch():
    """ctu_bn_finalize (training) + un-folded ctu_bn_relu_fwd -- the path taken only above BN_FOLD_MAX_VOXELS -- forced
    on a small tensor, with pooling, against nn.BatchNorm3d in training mode (values, running statistics after two
    updates, backward)."""
    import torch.nn as nn
    import torch.nn.functional as F
    import ctunet_b200.engine as E
    old = E.BN_FOLD_MAX_VOXELS
    E.BN_FOLD_MAX_VOXELS = 0
    try:
        for mode, tol in (("fp32", 1e-5), ("bf16", 2e-2)):
            g = torch.Generator().manual_seed(4)
            y = torch.randn(2, 7, 8, 16, 16, generator=g) * 2 + 0.5
            if mode == "bf16":
                y = y.to(torch.bfloat16).float()
            bn = nn.BatchNorm3d(7)
            with torch.no_grad():
                bn.weight.uniform_(0.5, 1.5, generator=g)
                bn.bias.uniform_(-0.3, 0.3, generator=g)
            bng = nn.BatchNorm3d(7).to(DEV)
            bng.load_state_dict(bn.state_dict())
            yr = y.clone().requires_grad_()
            ar = F.relu(bn(yr))
            pr = F.max_pool3d(ar, 2, 2)
            dA, dP = torch.randn(ar.shape, generator=g), torch.randn(pr.shape, generator=g)
            (ar * dA).sum().backward(retain_graph=True)
            (pr * dP).sum().backward()
            with torch.no_grad():
                bn(y)                                     # the checkpoint recomputation: second buffer update
            eng = E.Engine(torch.device(DEV), mode, record=True)
            ya = eng.pack(y.to(DEV))
            a, pooled = eng.bn_relu(ya, bng, True, extra_updates=1, pool=True)
            assert (eng.unpack(a).cpu() - ar.detach()).abs().max().item() <= tol * ar.abs().max().item()
            assert (eng.unpack(pooled).cpu() - pr.detach()).abs().max().item() <= tol * pr.abs().max().item()
            eng.agrads[id(a)] = eng.pack(dA.to(DEV))
            eng.agrads[id(pooled)] = eng.pack(dP.to(DEV))
            eng.run_tape()
            torch.cuda.synchronize()
            dy = eng.unpack(eng.agrads[id(ya)]).cpu()
            assert (dy - yr.grad).abs().max().item() <= max(tol, 1e-4) * 5 * yr.grad.abs().max().item()
            assert torch.allclose(eng.pgrads[id(bng.weight)].cpu(), bn.weight.grad, rtol=max(tol, 1e-4) * 5, atol=1e-3)
            assert torch.allclose(bng.running_mean.cpu(), bn.running_mean, rtol=1e-4, atol=1e-5)
            assert torch.allclose(bng.running_var.cpu(), bn.running_var, rtol=1e-4, atol=1e-5)
            assert int(bng.num_batches_tracked) == 2 == int(bn.num_batches_tracked)
    finally:
        E.BN_FOLD_MAX_VOXELS = old


@pytest.mark.parametrize("shape", [(2, 2, 32, 48, 64), (1, 2, 16, 32, 128)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_non_cubic_volumes(mode, shape):
    """D != H != W (tile selection uses h and w, chunking uses d): train step against the oracle."""
    from oracle import unet_oracle as O
    g = torch.Generator().manual_seed(5)
    x = (torch.rand(*shape, generator=g) > 0.7).float()
    sk = (torch.rand(shape[0], *shape[2:], generator=g) > 0.6).long()
    fl = ((torch.rand(shape[0], *shape[2:], generator=g) > 0.8) & (sk > 0)).long()
    oh = lambda t: torch.nn.functional.one_hot(t, 2).permute(0, 4, 1, 2, 3).float().contiguous()
    target = (oh(sk), oh(fl))
    sd, pn, ref_out, comps = _oracle_step("UNetSP", x, target)
    net, out, fake = _product_step("UNetSP", x, target, mode)
    tol = 1e-4 if mode == "fp32" else 2e-2
    for o, r in zip(out, ref_out):
        assert _relerr(o, r) < tol
    for k, v in comps.items():
        assert abs(fake.losses_and_metrics[k][0] - float(v)) < (1e-4 if mode == "fp32" else 5e-3), k
    if mode == "fp32":
        named = dict(net.named_parameters())
        for k in pn:
            if sd[k].grad is None or float(sd[k].grad.norm()) < 1e-5:
                continue
            rel = float((named[k].grad.cpu() - sd[k].grad).norm() / sd[k].grad.norm())
            assert rel < 2e-2, (k, rel)          # binary inputs: max-pool ties move a few entries (see test_gpu_models)


def test_captured_train_step_at_128_tracks_oracle_losses():
    """TrainStep(graph=True) -- the benchmarked driver -- on a 2 x 128^3 batch: three iterations of loss components
    against the fp32 oracle trained with torch.optim.Adam(amsgrad=True) on the same tensors."""
    from ctunet_b200.trainer import TrainStep
    from oracle import unet_oracle as O
    cfg = O.PRESETS["UNetSP"]
    x, (sk_t, fl_t) = O.make_training_batch(2, 2, 128, seed=1234)
    sd = O.build_state_dict(cfg, seed=0)
    pn = [k for k in sd if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))]
    for k in pn:
        sd[k].requires_grad_()
    opt = torch.optim.Adam([sd[k] for k in pn], lr=1e-3, amsgrad=True)
    net = _build("UNetSP")
    step = TrainStep(net, "double", 1.0, 1.0, lr=1e-3, graph=True)
    xg, tg = x.to(DEV), (sk_t.to(DEV), fl_t.to(DEV))
    for it in range(4):
        out = O.unet_forward(sd, x.clone().requires_grad_(), cfg, training=True)
        loss, comps = O.loss_double_output(out, (sk_t, fl_t), 1.0, 1.0)
        loss.backward()
        opt.step()
        for k in pn:
            sd[k].grad = None
        got = step(xg, tg).tolist()
        for u, v in zip(got, [float(c) for c in comps.values()]):
            assert abs(u - v) < 5e-3, (it, got, [float(c) for c in comps.values()])
    assert step._graph is not None


def test_sliding_window_128_patches_bf16_labels_match_oracle_away_from_ties():
    """BASELINE config 4 at the real patch size: two 128^3 patches of a phantom through the bf16 eval-mode network, gathered
    and labelled by the fused kernels, against the fp32 CPU oracle on the same patch grid.  Labels are bit-exact wherever
    the oracle's own decision margin |p1 - p0| exceeds the bf16 output tolerance (2e-2); the near-tie voxels are counted
    and reported, and the fp32 accumulate-check mode agrees on all but the exact-rounding ties."""
    import ctunet_b200 as C
    from ctunet_b200 import preprocess as P
    from oracle import unet_oracle as O
    cfg = O.PRESETS["UNetSP"]
    x, _ = O.make_training_batch(2, 2, 128, seed=4321)
    vol = torch.cat((x[0], x[1]), dim=3).contiguous()                  # [2, 128, 128, 256]: two patches side by side
    sd = O.build_state_dict(cfg, seed=0)
    with torch.no_grad():
        # Seed-0 weights decide every voxel with a wide margin (no ties at all): re-centre the head's bias on the median
        # logits so that both outputs are balanced decisions with a dense band of near-ties around the boundary --
        # skull = [s0, s1+s2] with s2 ~ 0 and s0, s1 ~ 0.5; flap = [1-s1, s1] with s1 ~ 0.5.
        probe = O.unet_forward(sd, vol[None, :, :, :, :128], O.UNetConfig(i_size=7, input_channels=2, out_channels=3), training=False)
        lc = torch.logit(probe.clamp(1e-6, 1 - 1e-6))[0]
        med = lc.flatten(1).median(dim=1).values
        sd["last_conv.bias"] = sd["last_conv.bias"] - med + torch.tensor([0.0, 0.0, -6.0])
        ref_outs = [O.unet_forward(sd, vol[None, :, :, :, i * 128:(i + 1) * 128], cfg, training=False) for i in range(2)]
    ref = [torch.cat([o[k][0] for o in ref_outs], dim=3) for k in range(2)]          # [2, 128, 128, 256] probabilities
    ref_lab = [torch.argmax(r, 0).float() for r in ref]
    margin = [(r[1] - r[0]).abs() for r in ref]
    for mode, tol in (("bf16", 2e-2), ("fp32", 1e-4)):
        C.set_compute_dtype(mode)
        torch.manual_seed(0)
        net = C.UNetSP()
        net.load_state_dict(sd)
        net = net.to(DEV).eval()
        C.set_compute_dtype("bf16")
        labs = P.sliding_window_argmax(net, vol.to(DEV), patch=128, batch=2)
        for k in range(2):
            lab = labs[k].cpu()
            assert lab.shape == (128, 128, 256)
            clear = margin[k] > tol
            mism = lab != ref_lab[k]
            assert not bool((mism & clear).any()), "%s output %d: a label differs where the margin is %.3g" % (
                mode, k, float(margin[k][mism & clear].max()))
            ones = float(ref_lab[k].mean())
            assert 0.05 < ones < 0.95, ones                    # a real decision boundary, not a constant label
            print("%s output %d: %.1f %% ones; %d of %d voxels within the %.0e tie band, %d of them labelled differently" % (
                mode, k, 100 * ones, int((~clear).sum()), clear.numel(), tol, int(mism.sum())))
