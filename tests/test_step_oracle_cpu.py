"""CPU checks of tests/step_oracle.py: the float64 optimizer and scheduler references against torch, the optimizer bound
against a float32 emulation of ``optim_step_kernel`` (and four wrong updates that must fall outside it), the flat-buffer
slot table against ``GradSync`` and the BatchNorm update counts."""
import math

import pytest
import torch

import step_oracle as S

HYPER = dict(beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, momentum=0.0, alpha=0.99, amsgrad=1)
CASES = [("adam", 0.0, 0.0), ("adam", 1e-2, 0.0), ("adamw", 1e-2, 0.0), ("rmsprop", 0.0, 0.0), ("rmsprop", 1e-2, 0.9),
         ("sgd", 0.0, 0.9), ("sgd", 1e-2, 0.0)]


def _hyper(wd, mom):
    return dict(HYPER, weight_decay=wd, momentum=mom)


def _grads(n, steps, seed):
    """Gradients over nine decades of magnitude, exact zeros and values whose squares are subnormal in fp32."""
    g = torch.Generator().manual_seed(seed)
    scale = 10.0 ** torch.randint(-9, 1, (n,), generator=g).double()
    out = []
    for _ in range(steps):
        t = torch.randn(n, generator=g, dtype=torch.float64) * scale
        t[::97] = 0.0
        t[5::101] *= 1e-12
        out.append(t.float().double())
    return out


def _init_states(kind, n):
    k = S.KIND_STATES[kind]
    return tuple(torch.zeros(n, dtype=torch.float64) if i < k else None for i in range(3))


def _kernel32(kind, p, g, states, lr, step, hp, bc_step=None, twice_m=False):
    """optim_step_kernel in float32 torch arithmetic (every operation rounded, no fused multiply-add).  ``bc_step``: the
    step number used for the bias corrections (default: the right one); ``twice_m``: m updated twice."""
    f = torch.float32
    p, g = p.float(), g.float()
    s = [t.float().clone() if t is not None else None for t in states]
    t = step + 1
    f32 = lambda v: torch.tensor(v, dtype=f)
    wd, mom = f32(hp["weight_decay"]), f32(hp["momentum"])
    lr32 = f32(lr)
    if kind in ("adam", "adamw"):
        tb = t if bc_step is None else bc_step
        ss = f32(lr / (1 - hp["beta1"] ** tb))
        bc2s = f32(math.sqrt(1 - hp["beta2"] ** tb))
        if hp["weight_decay"] != 0:
            if kind == "adam":
                g = p * wd + g
            else:
                p = p * (1 - lr32 * wd)
        omb1, omb2, b2 = f32(1 - hp["beta1"]), f32(1 - hp["beta2"]), f32(hp["beta2"])
        m = s[0] + (g - s[0]) * omb1
        if twice_m:
            m = m + (g - m) * omb1
        v = s[1] * b2 + omb2 * g * g
        vv = torch.maximum(s[2], v)
        denom = vv.sqrt() / bc2s + f32(hp["eps"])
        p = p - ss * (m / denom)
        out = (m, v, vv)
    elif kind == "rmsprop":
        if hp["weight_decay"] != 0:
            g = p * wd + g
        sq = s[0] * f32(hp["alpha"]) + f32(1 - hp["alpha"]) * g * g
        avg = sq.sqrt() + f32(hp["eps"])
        if hp["momentum"] > 0:
            buf = s[1] * mom + g / avg
            p = p - lr32 * buf
            out = (sq, buf, None)
        else:
            p = p - lr32 * (g / avg)
            out = (sq, None, None)
    else:
        if hp["weight_decay"] != 0:
            g = p * wd + g
        out = (None, None, None)
        if hp["momentum"] != 0:
            buf = g if t == 1 else s[0] * mom + g
            g = buf
            out = (buf, None, None)
        p = p - lr32 * g
    return p.double(), tuple(o.double() if o is not None else None for o in out)


@pytest.mark.parametrize("kind,wd,mom", CASES)
def test_optimizer_update64_equals_torch_optim_in_float64(kind, wd, mom):
    n, lr = 3000, 1e-3
    hp = _hyper(wd, mom)
    p0 = torch.randn(n, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    ref = p0.clone().requires_grad_()
    if kind in ("adam", "adamw"):
        cls = torch.optim.Adam if kind == "adam" else torch.optim.AdamW
        opt = cls([ref], lr=lr, betas=(hp["beta1"], hp["beta2"]), eps=hp["eps"], weight_decay=wd, amsgrad=True, foreach=False)
    elif kind == "rmsprop":
        opt = torch.optim.RMSprop([ref], lr=lr, alpha=hp["alpha"], eps=hp["eps"], weight_decay=wd, momentum=mom, foreach=False)
    else:
        opt = torch.optim.SGD([ref], lr=lr, momentum=mom, weight_decay=wd, foreach=False)
    p, st = p0.clone(), _init_states(kind, n)
    for k, g in enumerate(_grads(n, 5, 2)):
        ref.grad = g.clone()
        opt.step()
        up = S.optimizer_update64(kind, p, g, st, lr, k, hp)
        p, st = up.p, tuple(a if a is not None else b for a, b in zip(up.states, st))
        assert torch.equal(p, ref.detach()), (kind, k)
    tstate = opt.state[ref]
    names = {"adam": ("exp_avg", "exp_avg_sq", "max_exp_avg_sq"), "adamw": ("exp_avg", "exp_avg_sq", "max_exp_avg_sq"),
             "rmsprop": ("square_avg", "momentum_buffer"), "sgd": ("momentum_buffer",)}[kind]
    for i, nm in enumerate(names):
        if nm in tstate and tstate[nm] is not None:
            assert torch.equal(st[i], tstate[nm]), (kind, nm)


@pytest.mark.parametrize("kind,wd,mom", CASES)
def test_float32_kernel_emulation_stays_inside_the_bound(kind, wd, mom):
    n = 5000
    hp = _hyper(wd, mom)
    worst = 0.0
    for lr in (1e-4, 3e-2):
        p = (torch.randn(n, generator=torch.Generator().manual_seed(3), dtype=torch.float64) * 0.1).float().double()
        st = _init_states(kind, n)
        for k, g in enumerate(_grads(n, 12, 4)):
            up = S.optimizer_update64(kind, p, g, st, lr, k, hp)
            got_p, got_s = _kernel32(kind, p, g, st, lr, k, hp)
            err = (got_p - up.p).abs()
            assert bool((err <= up.p_err).all()), (kind, lr, k, float((err / up.p_err).max()))
            worst = max(worst, float((err / up.p_err).max()))
            for i in range(3):
                if up.states[i] is not None:
                    e = (got_s[i] - up.states[i]).abs()
                    assert bool((e <= up.state_errs[i]).all()), (kind, lr, k, i, float((e / up.state_errs[i]).max()))
            # continue from the fp32 kernel's own result, as the device does
            p = got_p
            st = tuple(a if a is not None else b for a, b in zip(got_s, st))
    print("%s wd=%g mom=%g: worst element at %.3f of its bound" % (kind, wd, mom, worst))
    assert worst > 0.01          # the bound is not vacuous: rounding errors reach a visible fraction of it


def test_wrong_adam_updates_fall_outside_the_bound():
    """Four ways a captured step can feed the optimizer wrongly, each outside the per-element bound."""
    n, lr = 4096, 1e-4
    hp = _hyper(0.0, 0.0)
    p = (torch.randn(n, generator=torch.Generator().manual_seed(5), dtype=torch.float64) * 0.1).float().double()
    st = _init_states("adam", n)
    grads = _grads(n, 6, 6)
    for k in range(4):
        p, st = _kernel32("adam", p, grads[k], st, lr, k, hp)
    k = 4
    g, g_prev = grads[k], grads[k - 1]
    up = S.optimizer_update64("adam", p, g, st, lr, k, hp)
    outside = lambda q: (q - up.p).abs() > up.p_err
    moved = (up.p - p).abs() > 1e3 * up.p_err                    # elements whose update is far above rounding
    assert float(moved.double().mean()) > 0.75
    # the gradient of the previous step
    bad, _ = _kernel32("adam", p, g_prev, st, lr, k, hp)
    assert float(outside(bad)[moved].double().mean()) > 0.9
    # one 1024-element chunk skipped (its parameters keep their value)
    bad, _ = _kernel32("adam", p, g, st, lr, k, hp)
    bad[2 * S.CHUNK:3 * S.CHUNK] = p[2 * S.CHUNK:3 * S.CHUNK]
    assert bool(outside(bad)[2 * S.CHUNK:3 * S.CHUNK][moved[2 * S.CHUNK:3 * S.CHUNK]].all())
    # the bias corrections of step k - 1
    bad, _ = _kernel32("adam", p, g, st, lr, k, hp, bc_step=k)
    assert bool(outside(bad)[moved].all())
    # m updated twice
    bad, bad_s = _kernel32("adam", p, g, st, lr, k, hp, twice_m=True)
    assert float(outside(bad)[moved].double().mean()) > 0.5
    assert float(((bad_s[0] - up.states[0]).abs() > up.state_errs[0]).double().mean()) > 0.9


def test_plateau64_equals_reduce_lr_on_plateau():
    cfg = dict(factor=0.5, patience=1, threshold=1e-3, min_lr=1e-5, cooldown=1, eps=1e-8)
    prm = torch.zeros(1, requires_grad=True)
    opt = torch.optim.SGD([prm], lr=1e-2)
    sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, **cfg)
    rec = torch.tensor([1e-2, math.inf, 0, 0, cfg["factor"], cfg["patience"], cfg["threshold"], cfg["min_lr"],
                        cfg["cooldown"], cfg["eps"]], dtype=torch.float64)
    losses = [1.0, 0.9, 0.8999, 0.95, 0.7, 0.7, 0.7, 0.6995, 0.69, 0.7, 0.71, 0.5, 0.5, 0.5, 0.5, 0.5]
    reductions = cooldowns = 0
    for x in losses:
        loss = torch.tensor(x, dtype=torch.float32)             # the device feeds the fp32 total
        old = rec[0].item()
        sch.step(loss)
        rec = S.plateau64(rec, loss)
        assert rec[0].item() == opt.param_groups[0]["lr"]
        assert rec[1].item() == sch.best
        assert rec[2].item() == sch.num_bad_epochs
        assert rec[3].item() == sch.cooldown_counter
        reductions += rec[0].item() < old
        cooldowns += rec[3].item() > 0
    assert reductions >= 2 and cooldowns >= 1


def _cpu_model(name):
    import ctunet_b200 as C
    torch.manual_seed(0)
    return getattr(C, name)()


@pytest.mark.parametrize("name", ["UNet", "UNet4b2i3o", "UNet5b2i3o", "UNet4b1i3o", "UNetSP", "UNetSPSmall", "UNetDO",
                                  "recAE_v2_fixed", "UNet4_2IC"])
def test_slot_table_equals_grad_sync_slices(name):
    from ctunet_b200.parallel import GradSync
    net = _cpu_model(name)
    sync = GradSync(net)
    got = [(n, sync.slices[id(p)].storage_offset(), sync.slices[id(p)].numel()) for n, p in zip(sync.names, sync.params)]
    table = S.slot_table(net)
    assert table == got
    assert sum(t[2] for t in table) == sync.n_grad
    shapes = dict((n, p.shape) for n, p in net.named_parameters())
    for n, p in zip(sync.names, sync.params):
        assert sync.slices[id(p)].shape == shapes[n]


@pytest.mark.parametrize("name", ["UNetSP", "recAE_v2_fixed"])
def test_bn_update_counts(name):
    """Every BatchNorm inside the reentrant checkpoint moves twice per step; the generic UNet's dead center block once."""
    counts = S.bn_update_counts(name)
    bns = {n for n, m in _cpu_model(name).named_modules() if isinstance(m, torch.nn.BatchNorm3d)}
    assert set(counts) == bns
    for k, v in counts.items():
        assert v == (1 if k.startswith("cblock.") else 2), (k, v)
