"""The benchmarked training step, replay by replay (GPU): ``TrainStep(net, handler, 1.0, 1.0, lr, scheduler, graph=True)``
in bf16 -- the forward, the fused head + loss, the backward on up to six streams, the deferred top-level weight gradients,
every parameter gradient in its slice of ``GradSync.flat``, the BatchNorm buffer updates on the leaf-tail stream, one
``ctu_optim_step`` and one ``ctu_optim_post`` -- checked after every replay of the captured graph:

  1. nothing non-finite in the gradients, the loss components, the parameters or the optimizer states;
  2. parameters and states = ``step_oracle.optimizer_update64`` of the state before the replay and the gradient the replay
     left in the flat buffer, within its per-element bound (an optimizer that read a slice before its producer wrote it
     leaves a parameter that does not match the final gradient);
  3. the step counter moves by one and the scheduler record is bit-equal to ``plateau64`` fed the replay's own total loss;
  4. gradients and loss components against a serial reference: the same network state run eagerly through
     ``TrainStep._forward_backward`` with every side stream and the weight-gradient deferral switched off, in a caching
     allocator filled with NaN.  Two such runs measure N_t, the per-tensor order noise of the fp32 atomics of the
     parameter-gradient reductions; the replay must sit within 4 N_t + 2^-20 max|g_ref| of the reference (the
     analytically zero biases in front of a BatchNorm: see ``_biases_before_batchnorm``);
  5. BatchNorm buffers: ``num_batches_tracked`` moves by ``bn_update_counts``, the running statistics equal the serial
     reference's to 2 fp32 ulps;
  6. on the first and the last replay at 128^3, the gradient read by parameter name through ``slot_table`` sits within
     ``step_oracle.noise_floor`` of the float oracles at the product's parameters (the only check that sees two
     same-shape parameters whose slices were swapped).

Before every replay the buffers the step must fully rewrite -- the gradient part of the flat buffer and the loss
components -- are filled with NaN.  After the last replay the state before it is copied back in place and the replay is
repeated: it passes every check above and matches what the first run of that replay wrote, directly (state that leaks
from one replay into the next outside the buffers named here would not).
"""
import contextlib
import math
import time

import pytest
import torch

import step_oracle as S

pytestmark = pytest.mark.gpu
DEV = "cuda"
ASYNC_FLAGS = ("WEIGHT_PREP_ASYNC", "WGRAD_ASYNC", "DEAD_BRANCH_ASYNC", "DEFER_BIG_WGRAD")
HANDLER = {"UNetSP": "double", "recAE_v2_fixed": "single"}
IN_CHANNELS = {"UNetSP": 2, "recAE_v2_fixed": 1}
BATCH_SEEDS = (11, 12, 13, 12, 14, 15)          # replay 4 sees replay 2's batch again
ANCHOR_REPLAYS = (1, len(BATCH_SEEDS))
# The noise-floor rule is established at 64^3 and above.  At 32^3 the deepest level holds 4^3 voxels per sample, where single
# ReLU and max-pool decisions move a BatchNorm gradient by more than the rule allows (measured: 0.036 against 0.025).
ANCHOR_MIN_SIZE = 64
ORDER_NOISE = 4.0
ABS_FLOOR = 2.0 ** -20


@contextlib.contextmanager
def _serial():
    """Every stage on the current stream in tape order: no weight-preparation, weight-gradient or dead-branch side
    stream, no deferred weight gradients."""
    import ctunet_b200.engine as E
    old = {f: getattr(E, f) for f in ASYNC_FLAGS}
    for f in ASYNC_FLAGS:
        setattr(E, f, False)
    try:
        yield
    finally:
        for f, v in old.items():
            setattr(E, f, v)


@contextlib.contextmanager
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _nan_fill_allocator():
    """Leave the caching allocator holding NaN in both of its pools: one large block, which the large buffers of the next
    eager step are carved from, and 400 blocks of 512 KB in the pool of 2 MB segments that serves requests of 1 MB or
    less.  A kernel that reads memory nobody wrote this step then reads NaN, whatever the buffer's size."""
    free, _ = torch.cuda.mem_get_info()
    big = torch.full((min(free // 2, 48 << 30) // 4,), float("nan"), dtype=torch.float32, device=DEV)
    small = [torch.full((128 * 1024,), float("nan"), dtype=torch.float32, device=DEV) for _ in range(400)]
    del big, small


@pytest.fixture(autouse=True)
def _release_cached_memory():
    """The NaN blocks stay reserved by this process's caching allocator: hand them back to the device after each test."""
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _build(name):
    import ctunet_b200 as C
    C.set_compute_dtype("bf16")
    torch.manual_seed(0)
    return getattr(C, name)().to(DEV)


def _batch(name, batch, size, seed):
    """(image, product target, one-hot target for the oracle) of one synthetic training batch on the device."""
    from ctunet_b200.synthetic import make_training_batch
    img, (sk, fl) = make_training_batch(batch, IN_CHANNELS[name], size, seed, device=DEV)
    if HANDLER[name] == "double":
        return img, tuple(t[:, 1].to(torch.uint8).contiguous() for t in (sk, fl)), (sk, fl)
    return img, sk, sk


def _flat_targets(t):
    return list(t) if isinstance(t, (tuple, list)) else [t]


def _bn_buffers(net):
    return {k: v for k, v in net.state_dict().items() if k.endswith(("running_mean", "running_var", "num_batches_tracked"))}


def _optim_states(step):
    o = step.optimizer
    return [o.state0, o.state1, o.state2]


def _snapshot(step):
    img, tgt = step.static_inputs()
    return dict(params={n: p.detach().clone() for n, p in step.model.named_parameters()},
                states=[s.clone() if s is not None else None for s in _optim_states(step)],
                sched=step.optimizer.sched.clone(), step_count=step.optimizer.step_count.clone(),
                bn={k: v.clone() for k, v in _bn_buffers(step.model).items()},
                inputs=[t.clone() for t in [img] + _flat_targets(tgt)])


def _restore(step, snap):
    """Copy a snapshot back into the step's own storages (the captured graph reads and writes those)."""
    with torch.no_grad():
        for n, p in step.model.named_parameters():
            p.copy_(snap["params"][n])
        for s, v in zip(_optim_states(step), snap["states"]):
            if s is not None:
                s.copy_(v)
        step.optimizer.sched.copy_(snap["sched"])
        step.optimizer.step_count.copy_(snap["step_count"])
        bufs = _bn_buffers(step.model)
        for k, v in snap["bn"].items():
            bufs[k].copy_(v)
        img, tgt = step.static_inputs()
        for d, v in zip([img] + _flat_targets(tgt), snap["inputs"]):
            d.copy_(v)


def _outputs(step):
    """Everything a replay writes, copied: gradients, loss components, parameters in slot order, states, counters and
    BatchNorm buffers."""
    o = step.optimizer
    return dict(flat=step.grads.flat[:step.grads.n_grad].clone(), comps=step._comps.clone(),
                params=torch.cat([dict(step.model.named_parameters())[nm].detach().reshape(-1)
                                  for nm, _, _ in S.slot_table(step.model)]),
                states=[s.clone() if s is not None else None for s in _optim_states(step)],
                sched=o.sched.clone(), step_count=o.step_count.clone(),
                bn={k: v.clone() for k, v in _bn_buffers(step.model).items()})


def _poison(step):
    step.grads.flat[:step.grads.n_grad].fill_(float("nan"))
    step._comps.fill_(float("nan"))


class _Serial:
    """The serial reference: a twin network loaded with the replay's starting state, one eager forward + loss + backward."""

    def __init__(self, name, lr, scheduler):
        from ctunet_b200.trainer import TrainStep
        self.net = _build(name)
        self.step = TrainStep(self.net, HANDLER[name], 1.0, 1.0, lr=lr, scheduler=scheduler, graph=False)

    def run(self, snap):
        sd = dict(snap["params"])
        sd.update(snap["bn"])
        self.net.load_state_dict(sd)
        img, *tgt = snap["inputs"]
        tgt = tuple(tgt) if len(tgt) > 1 else tgt[0]
        _poison(self.step)
        torch.cuda.synchronize()
        _nan_fill_allocator()
        with _serial():
            self.step._forward_backward(img, tgt)
        self.step.grads.begin_step()
        torch.cuda.synchronize()
        return dict(flat=self.step.grads.flat[:self.step.grads.n_grad].clone(), comps=self.step._comps.clone(),
                    bn={k: v.clone() for k, v in _bn_buffers(self.net).items()})


def _biases_before_batchnorm(net):
    """Names of the convolution biases that feed a BatchNorm directly (recAE_v2_fixed; the generic UNet's convolutions
    have none).  Their gradient is analytically zero: the kernels return the rounding residue of a sum of millions of
    bf16 terms that cancel, and the order of the fp32 atomics moves that residue by about 1e-5 of itself.  Two serial
    runs repeat one order bit for bit (N_t = 0) while a replay, whose blocks share the SMs with other streams, takes
    another one, so these slots are held to the size of the residue, max|g_ref|, instead of 4 N_t + 2^-20 max|g_ref|."""
    out = set()
    for prefix, m in net.named_modules():
        kids = list(m.named_children())
        for (n0, c0), (_, c1) in zip(kids, kids[1:]):
            if isinstance(c0, torch.nn.Conv3d) and isinstance(c1, torch.nn.BatchNorm3d) and c0.bias is not None:
                out.add("%s.%s.bias" % (prefix, n0) if prefix else n0 + ".bias")
    return out


def _ulps2(a, b):
    """2 fp32 ulps of the larger magnitude of a and b."""
    m = torch.maximum(a.abs(), b.abs()).float()
    return 2 * (torch.nextafter(m, torch.full_like(m, math.inf)) - m).double()


class _Checker:
    def __init__(self, name, step, serial):
        self.name, self.step, self.serial = name, step, serial
        self.slots = S.slot_table(step.model)
        self.residue = _biases_before_batchnorm(step.model)
        self.counts = S.bn_update_counts(name)
        self.worst = dict(optimizer=0.0, states=0.0, grads=0.0, comps=0.0, running=0.0, anchor=0.0)
        self.noise_rows = None
        self.grad_bound, self.comps_bound = {}, None

    def _ratio(self, key, err, bound):
        r = float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0
        self.worst[key] = max(self.worst[key], r)
        return r

    def references(self, snap):
        """Two serial runs from the snapshot: the reference and its order noise."""
        return self.serial.run(snap), self.serial.run(snap)

    def check(self, snap, refs, where):
        step = self.step
        ref, ref2 = refs
        n = step.grads.n_grad
        flat = step.grads.flat[:n]
        comps = step._comps
        params = dict(step.model.named_parameters())
        states = _optim_states(step)
        # 1. finite
        assert bool(torch.isfinite(flat).all()), "%s: a gradient slot is not finite (never written?)" % where
        assert bool(torch.isfinite(comps).all()), "%s: loss components %s" % (where, comps.tolist())
        for nm, p in params.items():
            assert bool(torch.isfinite(p).all()), "%s: parameter %s" % (where, nm)
        for i, s in enumerate(states):
            if s is not None:
                assert bool(torch.isfinite(s).all()), "%s: optimizer state%d" % (where, i)
        # 2. optimizer
        p0 = torch.cat([snap["params"][nm].reshape(-1) for nm, _, _ in self.slots])
        p1 = torch.cat([params[nm].detach().reshape(-1) for nm, _, _ in self.slots])
        lr, k = float(snap["sched"][0]), int(snap["step_count"])
        up = S.optimizer_update64(step.optimizer.kind, p0, flat, snap["states"], lr, k, step.optimizer.hyper)
        err = (p1.double() - up.p).abs()
        if bool((err > up.p_err).any()):
            i = int((err / up.p_err).argmax())
            nm = next(s[0] for s in self.slots if s[1] <= i < s[1] + s[2])
            raise AssertionError("%s: parameter %s element %d is %.3g from the optimizer reference, bound %.3g" % (
                where, nm, i, float(err[i]), float(up.p_err[i])))
        self._ratio("optimizer", err, up.p_err)
        for i, (s, ref_s, e_s) in enumerate(zip(states, up.states, up.state_errs)):
            if ref_s is None:
                continue
            e = (s.double() - ref_s).abs()
            assert bool((e <= e_s).all()), "%s: optimizer state%d off by %.3g of its bound" % (where, i, float((e / e_s).max()))
            self._ratio("states", e, e_s)
        for nm, p in params.items():                        # a parameter without a slot is never updated
            if not any(nm == s[0] for s in self.slots):
                assert torch.equal(p.detach(), snap["params"][nm]), "%s: %s has no gradient but moved" % (where, nm)
        # 3. counters
        assert int(step.optimizer.step_count) == k + 1, where
        want = S.plateau64(snap["sched"].cpu(), comps[-1].cpu())
        got = step.optimizer.sched.cpu()
        assert torch.equal(got, want), "%s: scheduler record %s, expected %s" % (where, got.tolist(), want.tolist())
        # 4. gradients and loss components against the serial reference
        rows = []
        for nm, off, cnt in self.slots:
            a, g1, g2 = flat[off:off + cnt], ref["flat"][off:off + cnt], ref2["flat"][off:off + cnt]
            noise = float((g1 - g2).abs().max())
            dist = float((a - g1).abs().max())
            bound = ORDER_NOISE * noise + ABS_FLOOR * float(g1.abs().max())
            if nm in self.residue:
                bound = max(bound, float(g1.abs().max()))
            rows.append((nm, float(g1.norm()), float(g1.abs().max()), noise, dist))
            self.grad_bound[nm] = bound
            assert dist <= bound, ("%s: gradient of %s is %.3g from the serial reference, bound %.3g (order noise N_t = %.3g, "
                                   "max|g| = %.3g)" % (where, nm, dist, bound, noise, float(g1.abs().max())))
            if bound > 0:
                self.worst["grads"] = max(self.worst["grads"], dist / bound)
        if self.noise_rows is None:
            self.noise_rows = rows
        c_ref, c_ref2 = ref["comps"].double(), ref2["comps"].double()
        c_err = (comps.double() - c_ref).abs()
        c_bound = torch.maximum(ORDER_NOISE * (c_ref - c_ref2).abs(), 2.0 ** -22 * c_ref.abs())
        self.comps_bound = c_bound
        assert bool((c_err <= c_bound).all()), "%s: loss components %s, serial %s" % (where, comps.tolist(), ref["comps"].tolist())
        self._ratio("comps", c_err, c_bound)
        # 5. BatchNorm buffers
        bufs = _bn_buffers(step.model)
        for key, v in bufs.items():
            if key.endswith("num_batches_tracked"):
                bn = key[:-len(".num_batches_tracked")]
                assert int(v) == int(snap["bn"][key]) + self.counts[bn], "%s: %s moved %d times" % (
                    where, bn, int(v) - int(snap["bn"][key]))
            else:
                e, b = (v.double() - ref["bn"][key].double()).abs(), _ulps2(v, ref["bn"][key])
                assert bool((e <= b).all()), "%s: %s is %.3g ulps from the serial reference" % (where, key, float((e / b * 2).max()))
                self._ratio("running", e, b)

    def same_as(self, orig, where):
        """The repeat of a replay against what the first run of that replay wrote (``_outputs``), directly: gradients and
        loss components within the bounds ``check`` just used for that replay, parameters and states bit-equal wherever
        the gradient is (the update is elementwise), counters bit-equal, running statistics within 2 fp32 ulps."""
        now = _outputs(self.step)
        equal = 0
        for nm, off, cnt in self.slots:
            a, b = now["flat"][off:off + cnt], orig["flat"][off:off + cnt]
            dist = float((a - b).abs().max())
            assert dist <= self.grad_bound[nm], "%s: gradient of %s is %.3g from the first run, bound %.3g" % (
                where, nm, dist, self.grad_bound[nm])
            equal += int(torch.equal(a, b))
        c_err = (now["comps"].double() - orig["comps"].double()).abs()
        assert bool((c_err <= self.comps_bound).all()), "%s: loss components %s, first run %s" % (
            where, now["comps"].tolist(), orig["comps"].tolist())
        same = now["flat"] == orig["flat"]
        assert torch.equal(now["params"][same], orig["params"][same]), "%s: parameters differ where the gradients do not" % where
        for i, (s, t) in enumerate(zip(now["states"], orig["states"])):
            if s is not None:
                assert torch.equal(s[same], t[same]), "%s: optimizer state%d differs where the gradients do not" % (where, i)
        assert torch.equal(now["sched"], orig["sched"]) and torch.equal(now["step_count"], orig["step_count"]), where
        for key, v in now["bn"].items():
            w = orig["bn"][key]
            if key.endswith("num_batches_tracked"):
                assert torch.equal(v, w), "%s: %s" % (where, key)
            else:
                assert bool(((v.double() - w.double()).abs() <= _ulps2(v, w)).all()), "%s: %s" % (where, key)
        return equal

    def anchor(self, snap, where, oracle_target):
        """The flat buffer by parameter name against the float oracles at the product's parameters."""
        step = self.step
        img = snap["inputs"][0]
        g = torch.Generator(device=DEV).manual_seed(99)
        xp = img * (1 + 3e-7 * torch.randn(img.shape, generator=g, device=DEV))
        sd = dict(snap["params"])
        sd.update(snap["bn"])
        with _no_tf32():
            bounds, _ = S.noise_floor(self.name, sd, img, xp, oracle_target)
        flat = step.grads.flat
        for nm, off, cnt in self.slots:
            ent = bounds[nm]
            assert ent is not None, "%s: %s has a gradient slot but no gradient in the oracle" % (where, nm)
            ref, bound, _ = ent
            if bound is None:
                continue
            err = S.rel_err(flat[off:off + cnt].view_as(ref), ref)
            assert err <= bound, "%s: gradient of %s is %.4f from the bf16 oracle, bound %.4f" % (where, nm, err, bound)
            self.worst["anchor"] = max(self.worst["anchor"], err / bound)


@pytest.mark.parametrize("name,batch,size,lr,scheduler", [
    ("UNetSP", 4, 128, 1e-4, True),
    ("recAE_v2_fixed", 4, 128, 1e-4, True),
    # patience 1 and a threshold of 0.5: every step after the first counts as bad unless it halves the loss (at the
    # default threshold this net improves at every step), so the learning rate drops every other step, replays included
    ("UNetSP", 2, 32, 3e-2, dict(patience=1, threshold=0.5)),
])
def test_captured_step_replays_match_float64_and_serial_references(name, batch, size, lr, scheduler):
    from ctunet_b200.trainer import GRAPH_WARMUP, TrainStep
    t0 = time.perf_counter()
    net = _build(name)
    step = TrainStep(net, HANDLER[name], 1.0, 1.0, lr=lr, scheduler=scheduler, graph=True)
    batches = {s: _batch(name, batch, size, s) for s in sorted(set(BATCH_SEEDS) | {10})}
    img, tgt, _ = batches[10]
    for _ in range(GRAPH_WARMUP + 1):                   # eager steps, then the capture (and its first replay)
        step(img, tgt)
    assert step._graph is not None
    serial = _Serial(name, lr, scheduler)
    chk = _Checker(name, step, serial)
    lrs = [float(step.optimizer.sched[0])]
    last = None
    for r, seed in enumerate(BATCH_SEEDS, 1):
        img, tgt, onehot = batches[seed]
        s_img, s_tgt = step.static_inputs()
        s_img.copy_(img)
        for d, v in zip(_flat_targets(s_tgt), _flat_targets(tgt)):
            d.copy_(v)
        snap = _snapshot(step)
        _poison(step)
        step(s_img, s_tgt)
        torch.cuda.synchronize()
        refs = chk.references(snap)
        chk.check(snap, refs, "%s replay %d" % (name, r))
        if r in ANCHOR_REPLAYS and size >= ANCHOR_MIN_SIZE:
            chk.anchor(snap, "%s replay %d" % (name, r), onehot)
        lrs.append(float(step.optimizer.sched[0]))
        last = (snap, refs, _outputs(step))
    # the last replay again, from its starting state copied back in place: checked like every replay, then against what
    # the first run of that replay wrote
    snap, refs, first = last
    _restore(step, snap)
    _poison(step)
    step(*step.static_inputs())
    torch.cuda.synchronize()
    where = "%s replay %d repeated" % (name, len(BATCH_SEEDS))
    chk.check(snap, refs, where)
    n_equal = chk.same_as(first, where)
    if isinstance(scheduler, dict):
        assert any(b < a for a, b in zip(lrs, lrs[1:])), "the scheduler never lowered the learning rate: %s" % lrs
    print("\n%s %dx%d^3, %d replays + 1 repeated, %.1f s; worst ratio to each bound: %s; learning rates %s; repeat: %d of "
          "%d gradient slots bit-equal to the first run" % (
              name, batch, size, len(BATCH_SEEDS), time.perf_counter() - t0,
              ", ".join("%s %.3f" % kv for kv in chk.worst.items()), ["%.3g" % v for v in lrs], n_equal, len(chk.slots)))
    print("order noise N_t of replay 1 (tensor, |g|_2, max|g|, N_t, distance of the replay):")
    for row in chk.noise_rows:
        print("  %-34s %10.4g %10.4g %10.3g %10.3g" % row)
