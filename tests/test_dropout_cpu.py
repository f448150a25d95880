"""CPU: Dropout3d support -- the dropout sites of every model class, the checkpoint layout, and the oracle's keep-factor
placement against the live reference (skipped when the reference is absent, as in tests/test_reference_live.py)."""
import pytest
import torch
import torch.nn.functional as F

import dropout_oracle as DO
from oracle import unet_oracle as O
from oracle.reference_loader import reference_available


@pytest.mark.parametrize("cls,n_sites", [("UNet", 8), ("UNetSP", 8), ("UNetSPSmall", 10), ("recAE_v2_fixed", 9),
                                         ("UNet4_2IC", 9)])
def test_dropout_sites_follow_the_block_batchnorms(cls, n_sites):
    import ctunet_b200 as C
    net = getattr(C, cls)()
    sites = net._dropout_sites()
    assert len(sites) == n_sites
    mods = dict(net.named_modules())
    for name, m, c in sites:
        assert mods[name] is m and isinstance(m, torch.nn.Dropout3d)
        parent, idx = name.rsplit(".", 1)
        bn = mods[parent + "." + str(int(idx) - 2)]               # Conv, BatchNorm, ReLU, Dropout3d
        assert isinstance(bn, torch.nn.BatchNorm3d) and bn.num_features == c
    assert "cblock.block.6" not in [s[0] for s in sites]           # the generic UNet's discarded center block
    assert net._dropout_config() == ()                             # presets: dropout_p = 0
    for _, m, _ in sites:
        m.p = 0.25
    net.train()
    assert net._dropout_config() == tuple((i, 0.25) for i in range(n_sites))
    sites[0][1].eval()                                             # a site in eval mode is the identity
    assert [i for i, _ in net._dropout_config()] == list(range(1, n_sites))
    net.eval()
    assert net._dropout_config() == ()
    assert net.dropout_keep("cuda:0") == {}                        # no pass has drawn masks yet


def test_state_dict_layout_does_not_change_with_dropout():
    import ctunet_b200 as C
    for a, b in ((C.UNet(dropout_p=0.3), C.UNet()), (C.recAE_v2_fixed(dropout_p=0.3), C.recAE_v2_fixed())):
        assert list(a.state_dict()) == list(b.state_dict())
        assert [k for k, _ in a.named_buffers()] == [k for k, _ in b.named_buffers()]


def test_oracle_keep_factors_of_one_are_the_identity():
    cfg = O.PRESETS["UNetSP"]
    sd = O.build_state_dict(cfg, seed=0)
    x = torch.rand(2, 2, 16, 16, 16, generator=torch.Generator().manual_seed(1))
    names = ["d_blocks.%d.block.6" % i for i in range(4)] + ["u_blocks.%d.block.7" % i for i in range(4)]
    chans = [7, 14, 28, 56, 56, 28, 14, 7]
    ones = {n: torch.ones(2, c) for n, c in zip(names, chans)}
    a = DO.unet_forward({k: v.clone() for k, v in sd.items()}, x, cfg, training=True)
    b = DO.unet_forward({k: v.clone() for k, v in sd.items()}, x, cfg, training=True, dropout_keep=ones)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    # with the bf16 storage points too (the keep factor is applied before the one rounding)
    a = DO.unet_forward({k: v.clone() for k, v in sd.items()}, x, cfg, training=True, act_round=torch.bfloat16)
    b = DO.unet_forward({k: v.clone() for k, v in sd.items()}, x, cfg, training=True, act_round=torch.bfloat16,
                        dropout_keep=ones)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert O._bn_relu.__module__ == O.__name__                    # the oracle is left as it was
    zero_top = dict(ones)
    zero_top["u_blocks.3.block.7"] = torch.zeros(2, 7)              # the last up block dropped: the head sees the skip only
    c = DO.unet_forward({k: v.clone() for k, v in sd.items()}, x, cfg, training=True, dropout_keep=zero_top)
    assert not torch.equal(a[0], c[0])


def _masks_of(ref_net):
    """Forward hooks on every Dropout3d: the [N, C] factor it applied (first call only -- the checkpoint recomputation
    repeats the same mask)."""
    masks, hooks = {}, []
    for name, m in ref_net.named_modules():
        if isinstance(m, torch.nn.Dropout3d):
            def hook(mod, inp, out, name=name):
                if name in masks:
                    return
                i, o = inp[0].detach(), out.detach()
                dropped = (o.abs().flatten(2).sum(2) == 0) & (i.abs().flatten(2).sum(2) > 0)
                k = torch.full(i.shape[:2], 1.0 / (1.0 - mod.p))
                k[dropped] = 0.0
                masks[name] = k
            hooks.append(m.register_forward_hook(hook))
    return masks, hooks


@pytest.mark.skipif(not reference_available(), reason="reference not present (run oracle/build_ref.py)")
@pytest.mark.parametrize("cls,cfg_name", [("UNet", "UNet"), ("recAE_v2_fixed", "recAE_v2_fixed")])
def test_oracle_with_reference_masks_equals_reference_training(cls, cfg_name):
    """The live reference with dropout_p = 0.3 in training mode; the masks its Dropout3d modules drew, fed to the oracle,
    reproduce its outputs and parameter gradients (the dropout sits after the block's second BatchNorm+ReLU, ahead of the
    max-pool and the skip)."""
    from oracle.reference_loader import load_reference
    MD = load_reference()[0]
    cfg = O.PRESETS[cfg_name]
    torch.manual_seed(0)
    ref = getattr(MD, cls)(dropout_p=0.3).train()
    sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
    g = torch.Generator().manual_seed(3)
    x = torch.rand(2, cfg.input_channels, 16, 16, 16, generator=g)
    wout = torch.randn(2, 2, 16, 16, 16, generator=g)
    masks, hooks = _masks_of(ref)
    torch.manual_seed(5)
    out = ref(x.clone().requires_grad_())
    out = out[0] if isinstance(out, tuple) else out
    (out * wout).sum().backward()
    for h in hooks:
        h.remove()
    assert any(float((k == 0).float().mean()) > 0 for k in masks.values())
    pn = [k for k in sd if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))]
    for k in pn:
        sd[k].requires_grad_()
    masks.pop("cblock.block.6", None)
    o2 = DO.unet_forward(sd, x.clone().requires_grad_(), cfg, training=True, dropout_keep=masks)
    o2 = o2[0] if isinstance(o2, tuple) else o2
    (o2 * wout).sum().backward()
    assert float((out - o2).abs().max()) <= 1e-5 * max(1.0, float(o2.abs().max()))
    named = dict(ref.named_parameters())
    for k in pn:
        if named[k].grad is None:
            continue
        gr = sd[k].grad
        assert float((named[k].grad - gr).abs().max()) <= 1e-5 * max(1.0, float(gr.abs().max())), k
