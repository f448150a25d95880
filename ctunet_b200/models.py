"""Drop-in replacements for ``ctunet.pytorch.models`` (reference: ctunet/pytorch/models.py).

Same class names, constructor signatures, attributes, ``state_dict`` layout (SURVEY.md Appendix B)
and ``forward`` return structure as the reference, so that ``eval(model_class)()`` in
``ctunet/pytorch/Model.py:485,488`` can resolve to these classes.  The sub-modules
(``nn.Conv3d`` / ``nn.BatchNorm3d`` / ``nn.ConvTranspose3d``) are kept purely as parameter
containers: constructing them in the reference's order gives identical same-seed initialisation
and identical checkpoint keys.  The arithmetic never goes through them -- ``forward`` runs the fused
sm_100a kernels through the C ABI (engine.py), and raises for non-CUDA inputs (no CPU fallback).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib
from .engine import DropoutRNG, Engine

_COMPUTE_DTYPE = "bf16"


def set_compute_dtype(mode: str) -> None:
    """'bf16' (product mode: bf16 activations, fp32 accumulation) or 'fp32' (accumulate-check mode).
    Applies to models constructed afterwards; an existing model can be switched via ``.compute_dtype``."""
    global _COMPUTE_DTYPE
    if mode not in ("bf16", "fp32"):
        raise ValueError("mode must be 'bf16' or 'fp32'")
    _COMPUTE_DTYPE = mode


def get_compute_dtype() -> str:
    return _COMPUTE_DTYPE


def _only_inside_unet(self, x):
    raise NotImplementedError(
        "%s is a parameter container of the fused B200 path; it only executes inside UNet.forward / "
        "recAE_v2_fixed.forward" % type(self).__name__)


class UNetBlock(nn.Module):
    """models.py:9-49 -- conv-bn-relu x2 (+ConvTranspose3d first when up_block)."""

    def __init__(self, in_c, out_c, kern_s_conv=5, kern_s_uconv=2, pad=2, stride_c=1, stride_upc=2, dropout_p=0,
                 up_block=False):
        super().__init__()
        if not up_block:
            self.block = nn.Sequential(
                nn.Conv3d(in_c, out_c, kern_s_conv, stride_c, pad, bias=False),
                nn.BatchNorm3d(out_c),
                nn.ReLU(True),
                nn.Conv3d(out_c, out_c, kern_s_conv, stride_c, pad, bias=False),
                nn.BatchNorm3d(out_c),
                nn.ReLU(True),
                nn.Dropout3d(dropout_p))
        else:
            self.block = nn.Sequential(
                nn.ConvTranspose3d(in_c, in_c, kern_s_uconv, stride_upc),
                nn.Conv3d(in_c, out_c, kern_s_conv, stride_c, pad, bias=False),
                nn.BatchNorm3d(out_c),
                nn.ReLU(True),
                nn.Conv3d(out_c, out_c, kern_s_conv, stride_c, pad, bias=False),
                nn.BatchNorm3d(out_c),
                nn.ReLU(True),
                nn.Dropout3d(dropout_p))

    forward = _only_inside_unet


class CenterBlock(nn.Module):
    """models.py:52-97 (convolutional variant; the fully-connected variants are never used by a
    live model class and are not provided)."""

    def __init__(self, input_channels, output_channels, kern_sz_conv, padding, dropout_p, fc_block=False):
        super().__init__()
        if fc_block:
            raise NotImplementedError("CenterBlock fc_block variants (models.py:83-94) are outside the hot path")
        self.block = nn.Sequential(
            nn.Conv3d(input_channels, output_channels, kern_sz_conv, padding=padding, bias=False),
            nn.BatchNorm3d(output_channels),
            nn.ReLU(True),
            nn.Conv3d(output_channels, output_channels, kern_sz_conv, padding=padding, bias=False),
            nn.BatchNorm3d(output_channels),
            nn.ReLU(True),
            nn.Dropout3d(dropout_p))

    forward = _only_inside_unet


class ResidualBlock(nn.Module):
    """models.py:100-155 -- reachable only through UNet(residual=True); no live preset uses it."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        raise NotImplementedError("ResidualBlock (UNet(residual=True)) is outside the hot path (SURVEY.md 8a, row a4)")


def _check_conv_geometry(k, pad, stride=1):
    if k not in (1, 3, 5) or pad != k // 2 or stride != 1:
        raise NotImplementedError(
            "the fused path covers Conv3d with kernel 1/3/5, stride 1 and 'same' padding (got k=%d pad=%d stride=%d)"
            % (k, pad, stride))


def _up_stage(eng: Engine, srcs, ct: nn.ConvTranspose3d, cv: nn.Conv3d, k: int, training: bool):
    """ConvTranspose3d(k2, s2) + the first Conv3d of an up block (models.py:37-38, :427-430): one composed
    convolution on the low-resolution grid where the engine covers it, the two separate stages otherwise."""
    if eng.up_fusable(srcs, cv.weight.shape[0], k):
        return eng.up_conv(srcs, ct, cv, k, [True] * len(srcs), training)
    t = eng.convt(srcs, ct.weight, ct.bias, [True] * len(srcs))
    return eng.conv([t], cv.weight, cv.bias, k, [True], training)


class _FusedNet(nn.Module):
    """Common forward driver: validates the input, runs the engine, wires autograd."""

    compute_dtype: str

    def _levels(self) -> int:
        raise NotImplementedError

    def _run(self, eng: Engine, x: torch.Tensor, training: bool):
        raise NotImplementedError

    # ---- Dropout3d (the last module of every block, models.py:34,46,97,411,438,492)
    def _dropout_sites(self):
        """[(name, nn.Dropout3d, channels)] of the dropout sites whose input the network uses, in a fixed order: the index
        is the site's number in the Philox counter of its keep factors (csrc/dropout.cu)."""
        raise NotImplementedError

    def _active_dropout(self):
        """Sites that drop in this pass: read from each site's own module like torch does (``.training`` and ``.p``), so
        an eval-mode net with its Dropout3d modules switched to train draws masks too (Monte-Carlo dropout inference)."""
        return [(i, name, m, c) for i, (name, m, c) in enumerate(self._dropout_sites()) if m.training and m.p > 0]

    def _dropout_config(self):
        """What a captured graph / weight-preparation plan of a pass depends on: (site, p) of every active site."""
        return tuple((i, float(m.p)) for i, _, m, _ in self._active_dropout())

    def _draw_dropout(self, eng: Engine, n: int):
        """Keep factors of every active site for this pass (one launch beside the layer chain): {site name: [n, cpad]}."""
        act = self._active_dropout()
        if not act:
            return {}
        # a plain attribute, not a buffer: the state_dict / checkpoint layout stays the reference's.  nn.DataParallel
        # replicas share the dict (a shallow copy of __dict__), so every device keeps its state across steps.
        states = self.__dict__.setdefault("_dropout_rng", {})
        key = str(eng.device)
        rng = states.get(key)
        if rng is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("the first pass that draws dropout masks on %s is being captured in a CUDA graph: run "
                                   "it eagerly once first (its random state is created then)" % key)
            rng = states[key] = DropoutRNG(eng.device)
        views = eng.dropout_masks(rng, n, [(i, c, float(m.p)) for i, _, m, c in act])
        rng.last = {name: v[:, :c] for (_, name, _, c), v in zip(act, views)}
        return {name: v for (_, name, _, _), v in zip(act, views)}

    def dropout_keep(self, device=None):
        """{Dropout3d module name: float32 [N, C] keep factors} of the last pass that drew masks on ``device`` (default:
        the parameters' device): 0 for a dropped channel, 1/(1-p) for a kept one.  Views of the pass's own buffer, valid
        until the next forward; after a replay of a captured step they hold that replay's masks."""
        if device is None:
            device = self._weight_tensors()[0].device
        rng = self.__dict__.get("_dropout_rng", {}).get(str(torch.device(device)))
        return dict(rng.last) if rng is not None else {}

    def _validate(self, x: torch.Tensor):
        if not isinstance(x, torch.Tensor) or x.dim() != 5:
            raise ValueError("expected a 5-D [B, C, D, H, W] tensor")
        if not x.is_cuda:
            raise RuntimeError("ctunet_b200 runs on CUDA (sm_100a) only: there is no CPU fallback; got a %s tensor"
                               % x.device.type)
        if x.dtype != torch.float32:
            raise TypeError("expected float32 input (the reference feeds float32 NCDHW), got %s" % x.dtype)
        m = 2 ** self._levels()
        if any(s % m for s in x.shape[2:]):
            raise ValueError("spatial size %s must be divisible by %d" % (tuple(x.shape[2:]), m))
        for p in self._weight_tensors():
            if p.device != x.device or p.dtype != torch.float32:
                raise RuntimeError("parameters must be float32 on %s (call .to(device))" % x.device)
            break

    def _weight_tensors(self):
        """The tensors the engine reads through the parameter containers, in ``named_parameters`` order.  On an
        ``nn.DataParallel`` replica (Model.py:486; torch.nn.parallel.replicate) ``parameters()`` is EMPTY: the broadcast
        copies are plain attributes listed in ``_former_parameters`` -- non-leaf tensors whose gradients flow back to the
        real parameters through the Broadcast node, so they must be inputs of the autograd function like parameters."""
        if not getattr(self, "_is_replica", False):
            return list(self.parameters())
        out = []
        for m in self.modules():
            out.extend(t for t in getattr(m, "_former_parameters", {}).values() if t is not None)
        return out

    def forward(self, x):
        self._validate(x)
        x = x.contiguous()
        params = self._weight_tensors()
        record = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        if not record:
            eng = Engine(x.device, self.compute_dtype, record=False)
            return _run_planned(self, eng, x, False, params)
        if DROPIN_GRAPH and self.training and not getattr(self, "_is_replica", False) and getattr(self, "_grad_sink", None) is None:
            return _GraphNetFn.apply(self, x, *params)
        return _NetFn.apply(self, x, *params)


    @torch.no_grad()
    def predict_labels(self, x=None, *, vol=None, origins=None, patch=None, out=None):
        """The 'test' branch of the reference (Model.py:376-380 + ProblemHandler.py:338-343): eval-mode forward and
        ``hard_segm_from_tensor`` of every output, as float32 label volumes -- the head kernel writes the labels itself.
        Either ``x`` [B,C,D,H,W] (labels [B,D,H,W] per output), or sliding-window mode: ``vol`` float32 [C,D,H,W] on the device,
        ``origins`` device int32 [B,3] (z, y, x) and ``patch``: the B patches are gathered from ``vol`` by one kernel and
        their labels scattered into the full-size volumes ``out`` (a list of float32 [D,H,W] tensors, one per output)."""
        was = self.training
        self.eval()
        try:
            params = self._weight_tensors()
            if vol is None:
                self._validate(x)
                x = x.contiguous()
                eng = Engine(x.device, self.compute_dtype, record=False)
                n_out = 2 if getattr(self, "_head_mode", "plain") != "plain" else 1
                labels = [torch.empty((x.shape[0],) + tuple(x.shape[2:]), dtype=torch.float32, device=x.device) for _ in range(n_out)]
                eng.label_dst = (labels, None, 0, None)
                _run_planned(self, eng, x, False, params)
                return tuple(labels)
            if not (vol.is_cuda and vol.dtype == torch.float32 and vol.dim() == 4 and vol.is_contiguous()):
                raise TypeError("vol: contiguous float32 CUDA tensor [C, D, H, W]")
            if not (origins.is_cuda and origins.dtype == torch.int32 and origins.dim() == 2 and origins.shape[1] == 3):
                raise TypeError("origins: CUDA int32 tensor [B, 3]")
            m = 2 ** self._levels()
            if patch % m or patch % 4 or vol.shape[3] % 4:
                raise ValueError("patch size %d must be divisible by %d (and the volume width by 4)" % (patch, max(m, 4)))
            eng = Engine(vol.device, self.compute_dtype, record=False)
            eng.patch_src = (vol, origins.contiguous(), int(patch))
            eng.label_dst = (list(out), origins.contiguous(), int(patch), tuple(vol.shape[1:]))
            shape = torch.empty((origins.shape[0], vol.shape[0], patch, patch, patch), device="meta")
            _run_planned(self, eng, shape, False, params, device=vol.device)
            return tuple(out)
        finally:
            self.train(was)

    @torch.no_grad()
    def accumulate_windows(self, *, vol, origins, patch, weights, acc):
        """Overlapping sliding-window mode (preprocess.sliding_window_predict): eval-mode forward of the B windows of
        ``patch``^3 voxels at the device int32 ``origins`` [B,3] (z, y, x; anywhere: input voxels outside ``vol`` read as 0),
        gathered from ``vol`` float32 [C,D,H,W], and every window voxel inside the volume adds its weighted head outputs to
        the int64 accumulators ``acc`` [n_out * channels, D, H, W] in 2^-40 fixed point.  ``weights`` is the device
        float32 [3, patch] table of the separable window weight.  Returns ``acc``."""
        was = self.training
        self.eval()
        try:
            if not (vol.is_cuda and vol.dtype == torch.float32 and vol.dim() == 4 and vol.is_contiguous()):
                raise TypeError("vol: contiguous float32 CUDA tensor [C, D, H, W]")
            if not (origins.is_cuda and origins.dtype == torch.int32 and origins.dim() == 2 and origins.shape[1] == 3):
                raise TypeError("origins: CUDA int32 tensor [B, 3]")
            if not (weights.is_cuda and weights.dtype == torch.float32 and tuple(weights.shape) == (3, patch)):
                raise TypeError("weights: CUDA float32 tensor [3, patch]")
            if not (acc.is_cuda and acc.dtype == torch.int64 and acc.is_contiguous() and acc.shape[1:] == vol.shape[1:]):
                raise TypeError("acc: contiguous int64 CUDA tensor [n_out * channels, D, H, W]")
            m = 2 ** self._levels()
            if patch % m or patch % 4:
                raise ValueError("patch size %d must be divisible by %d" % (patch, max(m, 4)))
            eng = Engine(vol.device, self.compute_dtype, record=False)
            eng.patch_src = (vol, origins.contiguous(), int(patch))
            eng.accum_dst = (acc, origins.contiguous(), int(patch), tuple(vol.shape[1:]), weights.contiguous())
            shape = torch.empty((origins.shape[0], vol.shape[0], patch, patch, patch), device="meta")
            _run_planned(self, eng, shape, False, params=self._weight_tensors(), device=vol.device)
            return acc
        finally:
            self.train(was)


def _run_planned(net, eng: Engine, x, record: bool, params, device=None):
    """Run the network with the weight-preparation plan of this (shape, mode) configuration (Engine.begin).
    A plan holds closures over the weight tensors seen when it was recorded, so it is only reused while the module still
    owns the very same tensor objects (checked by identity against strong references kept with the plan: a parameter
    replaced by ``load_state_dict(assign=True)``, a swapped ``last_conv``, ... invalidates it); DataParallel replicas,
    whose tensors are new on every forward, never use plans."""
    from . import engine as E
    if getattr(net, "_is_replica", False):
        out = net._run(eng, x, net.training)
        eng.end_forward()
        return out
    store = net.__dict__.setdefault("_prep_plans", {})
    key = (tuple(x.shape), str(device if device is not None else x.device), net.compute_dtype, bool(net.training), record,
           eng.want_input_grad, E.UP_FUSION, E.CONV_PATH, eng.patch_src is not None, eng.label_dst is not None,
           net._dropout_config(), eng.accum_dst is not None)
    owners = store.setdefault("__owners__", {})
    held = owners.get(key)
    if held is None or len(held) != len(params) or any(a is not b for a, b in zip(held, params)):
        store.pop(key, None)
        owners[key] = list(params)
    eng.begin(store, key)
    out = net._run(eng, x, net.training)
    eng.end_forward()
    return out


class _NetFn(torch.autograd.Function):
    """The whole network as one autograd node (forward tape recorded by the engine)."""

    @staticmethod
    def forward(ctx, net, x, *params):
        eng = Engine(x.device, net.compute_dtype, record=True)
        eng.grad_sink = getattr(net, "_grad_sink", None)
        eng.want_input_grad = bool(ctx.needs_input_grad[1])
        out = _run_planned(net, eng, x, True, params)
        ctx.eng = eng
        ctx.params = params
        ctx.two = isinstance(out, tuple)
        return out

    @staticmethod
    def backward(ctx, *gouts):
        eng = ctx.eng
        if eng is None:
            raise RuntimeError("the fused U-Net graph was already freed (backward called twice)")
        g = [None if go is None else go.contiguous().float() for go in gouts]
        eng.backward(g[0], g[1] if ctx.two else None)
        dx = None
        if eng.want_input_grad:
            dx = eng.input_grad if eng.input_grad is not None else eng.unpack(eng.agrads.pop(id(eng.input_act)))
        if eng.grad_sink is not None:
            # gradients were written into the data-parallel flat buffer; GradSync.finish() publishes them
            grads = tuple(None if eng.grad_sink.buffer_for(p) is not None else
                          (eng.pgrads.get(id(p)) if p.requires_grad else None) for p in ctx.params)
        else:
            grads = tuple(eng.pgrads.get(id(p)) if p.requires_grad else None for p in ctx.params)
        ctx.eng = None
        return (None, dx) + grads


# Opt-in (``ctunet_b200.install(graph=True)``): the autograd node replays CAPTURED forward / backward graphs.  Behind the
# reference's own step driver (Model.forward_pass) the eager launch stream is host-bound (~7 ms of Python for 4.2 ms of
# kernels); the loss handler, torch.optim and the scheduler stay eager, as the reference drives them.
DROPIN_GRAPH = False
DROPIN_GRAPH_WARMUP = 2


class _GraphState:
    __slots__ = ("calls", "x", "out", "eng", "fwd", "bwd", "gouts", "dx", "grads", "two", "pending", "owners")

    def __init__(self):
        self.calls = 0
        self.fwd = self.bwd = self.eng = None
        self.pending = False


class _GraphNetFn(torch.autograd.Function):
    """``_NetFn`` with the forward pass and the backward pass each replayed from a CUDA graph captured on the third call
    of a (shape, mode) configuration.  The two graphs share one memory pool: the activations the backward tape reads are
    the forward graph's own allocations.  Restrictions (each falls back to the eager node): DataParallel replicas, a
    gradient sink, a second training forward before the backward of the first, parameters replaced after the capture."""

    @staticmethod
    def forward(ctx, net, x, *params):
        from . import engine as E
        store = net.__dict__.setdefault("_dropin_graphs", {})
        want_dx = bool(ctx.needs_input_grad[1])
        key = (tuple(x.shape), str(x.device), net.compute_dtype, want_dx, E.UP_FUSION, E.CONV_PATH, net._dropout_config())
        st = store.get(key)
        if st is None:
            st = store[key] = _GraphState()
        stale = st.fwd is not None and (len(st.owners) != len(params) or any(a is not b for a, b in zip(st.owners, params)))
        if stale:
            st = store[key] = _GraphState()
        ctx.st = None
        if st.pending or (st.fwd is None and st.calls < DROPIN_GRAPH_WARMUP):
            st.calls += 1
            return _NetFn.forward(ctx, net, x, *params)             # eager (warm-up / nested use)
        if st.fwd is None:
            st.x = torch.empty_like(x)
            st.x.copy_(x)
            st.owners = list(params)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=E.chain_stream(x.device)):
                eng = Engine(x.device, net.compute_dtype, record=True)
                eng.want_input_grad = want_dx
                out = _run_planned(net, eng, st.x, True, params)
            st.eng, st.fwd = eng, g
            st.two = isinstance(out, tuple)
            st.out = out if st.two else (out,)
            g.replay()
        else:
            st.x.copy_(x, non_blocking=True)
            st.fwd.replay()
        st.pending = True
        ctx.st = st
        ctx.params = params
        outs = tuple(o.detach() for o in st.out)                     # aliases of the static outputs (fresh autograd identities)
        return outs if st.two else outs[0]

    @staticmethod
    def backward(ctx, *gouts):
        from . import engine as E
        st = ctx.st
        if st is None:
            return _NetFn.backward(ctx, *gouts)
        g = [None if go is None else go.contiguous().float() for go in gouts]
        if st.bwd is None:
            st.gouts = [None if t is None else t.clone() for t in g]
            torch.cuda.synchronize()
            g2 = torch.cuda.CUDAGraph()
            eng = st.eng
            with torch.cuda.graph(g2, pool=st.fwd.pool(), stream=E.chain_stream(st.x.device)):
                eng.backward(st.gouts[0], st.gouts[1] if st.two else None)
                st.dx = None
                if eng.want_input_grad:
                    st.dx = eng.input_grad if eng.input_grad is not None else eng.unpack(eng.agrads.pop(id(eng.input_act)))
                st.grads = tuple(eng.pgrads.get(id(p)) if p.requires_grad else None for p in ctx.params)
            st.bwd = g2
            g2.replay()
        else:
            for dst, src in zip(st.gouts, g):
                if (dst is None) != (src is None):
                    raise RuntimeError("graph drop-in: the set of outputs that receive a gradient changed after the capture")
                if dst is not None:
                    dst.copy_(src, non_blocking=True)
            st.bwd.replay()
        st.pending = False
        ctx.st = None
        # (AccumulateGrad copies these: the static buffers stay owned by the graph)
        return (None, st.dx) + tuple(st.grads)


class UNet(_FusedNet):
    """U-Net generic model (models.py:158-261)."""

    def __init__(self, input_channels=1, out_channels=2, n_blocks=4, kern_sz_conv=3, kern_sz_upconv=2, stride_conv=1,
                 stride_upconv=2, i_size=8, padding=1, dropout_p=0, use_checkpoint=True, fc_layer=None,
                 use_skip_connections=True, apply_softmax=False, apply_sigmoid=True, cat=True, residual=False):
        super().__init__()
        self.chk = use_checkpoint
        self.skip = use_skip_connections
        self.apply_softmax = apply_softmax
        self.apply_sigmoid = apply_sigmoid
        self.fc_layer = fc_layer
        self.cat = cat
        self.compute_dtype = _COMPUTE_DTYPE
        self._head_mode = "plain"
        if residual:
            raise NotImplementedError("UNet(residual=True) is outside the hot path (SURVEY.md 8a, row a4)")
        if fc_layer:
            raise NotImplementedError("UNet(fc_layer=...) is outside the hot path (no live preset uses it)")
        if not cat and use_skip_connections:
            raise NotImplementedError("UNet(cat=False) (additive skips) is outside the hot path")
        if kern_sz_upconv != 2 or stride_upconv != 2:
            raise NotImplementedError("the fused path covers ConvTranspose3d kernel 2 / stride 2 only")
        _check_conv_geometry(kern_sz_conv, padding, stride_conv)
        self._k = kern_sz_conv
        self._dropout_p = dropout_p
        self._dropout_rng = {}        # device -> engine.DropoutRNG (created by the first pass that draws masks there)

        self.mp = nn.MaxPool3d(kernel_size=2, padding=0, stride=2, dilation=1, return_indices=True)
        d_blocks, u_blocks = [], []
        for i in range(n_blocks):                                                   # models.py:196-201
            c1 = input_channels if i == 0 else i_size * pow(2, i - 1)
            c2 = i_size * pow(2, i)
            d_blocks.append(UNetBlock(c1, c2, kern_sz_conv, 0, padding, stride_conv, 0, dropout_p))
        self.d_blocks = nn.ModuleList(d_blocks)
        icb, ocb = i_size * pow(2, n_blocks - 1), i_size * pow(2, n_blocks)
        self.cblock = CenterBlock(icb, ocb, kern_sz_conv, padding, dropout_p, fc_layer)   # models.py:204-206
        for i in range(n_blocks - 1, -1, -1):                                       # models.py:208-220
            if self.skip or i == n_blocks - 1:
                c1 = i_size * pow(2, i) * (2 if i == (n_blocks - 1) else 4)
                c1 = c1 // 2 if (self.fc_layer and i == (n_blocks - 1)) else c1
                c1 = c1 // 2 if not self.cat or (i == n_blocks - 1) else c1
                c2 = int(i_size * pow(2, i))
            else:
                c1 = i_size * pow(2, i) * 2
                c2 = i_size * pow(2, i)
            u_blocks.append(UNetBlock(c1, c2, kern_sz_conv, kern_sz_upconv, padding, stride_conv, stride_upconv,
                                      dropout_p, True))
        self.u_blocks = nn.ModuleList(u_blocks)
        lc_in = 2 * i_size if (self.skip and self.cat) else i_size
        self.last_conv = nn.Conv3d(lc_in, out_channels, 1)                          # models.py:223-224

    def _levels(self):
        return len(self.d_blocks)

    def _dropout_sites(self):
        # (the center block's Dropout3d is not a site: its output is discarded, models.py:238-241, DESIGN.md section 1)
        return ([("d_blocks.%d.block.6" % i, b.block[6], b.block[4].num_features) for i, b in enumerate(self.d_blocks)]
                + [("u_blocks.%d.block.7" % i, b.block[7], b.block[5].num_features) for i, b in enumerate(self.u_blocks)])

    def _head_flags(self):
        f = 0
        if self.apply_softmax:
            f |= _lib.HEAD_SOFTMAX
        if self.apply_sigmoid:
            f |= _lib.HEAD_SIGMOID
        if self._head_mode == "sp":
            f |= _lib.HEAD_SP
        elif self._head_mode == "sp_softmax":
            f |= _lib.HEAD_SP_SOFTMAX
        return f

    def _run(self, eng: Engine, x, training):
        """UNet.forward (models.py:226-261) as fused stages."""
        k = self._k
        extra = 1 if self.chk else 0          # checkpoint recomputation: one more BN buffer update at backward
        cur = eng.pack(x)
        eng.input_act = cur
        keep = self._draw_dropout(eng, x.shape[0])
        skips = []
        for i, blk in enumerate(self.d_blocks):
            seq = blk.block
            y = eng.conv([cur], seq[0].weight, seq[0].bias, k, [eng.want_input_grad if i == 0 else True], training,
                         leaf_input=(i == 0))
            a = eng.bn_relu(y, seq[1], training, extra)
            y = eng.conv([a], seq[3].weight, seq[3].bias, k, [True], training)
            s, cur = eng.bn_relu(y, seq[4], training, extra, pool=True,        # skip tensor + MaxPool (models.py:233)
                                 keep=keep.get("d_blocks.%d.block.6" % i))
            skips.append(s)
        if training:
            # models.py:238-241 -- the center block runs (its BatchNorm buffers move once) and its output is
            # discarded: no gradient ever reaches it.
            rec, eng.record = eng.record, False
            seq = self.cblock.block
            with eng.off_critical_path(cur):
                y = eng.conv([cur], seq[0].weight, seq[0].bias, k, [False], True)
                a = eng.bn_relu(y, seq[1], True)
                y = eng.conv([a], seq[3].weight, seq[3].bias, k, [False], True)
                eng.bn_relu(y, seq[4], True)
            eng.record = rec
        srcs = [cur]
        for i, blk in enumerate(self.u_blocks):
            seq = blk.block
            y = _up_stage(eng, srcs, seq[0], seq[1], k, training)
            a = eng.bn_relu(y, seq[2], training, extra)
            y = eng.conv([a], seq[4].weight, seq[4].bias, k, [True], training)
            ubl = eng.bn_relu(y, seq[5], training, extra, keep=keep.get("u_blocks.%d.block.7" % i))
            srcs = [ubl, skips[-i - 1]] if self.skip else [ubl]                  # models.py:247-253 (cat folded)
        return eng.head(srcs, self.last_conv.weight, self.last_conv.bias, self._head_flags())


class UNet4b2i3o(UNet):
    """models.py:272-278"""

    def __init__(self):
        super().__init__(i_size=7, input_channels=2, out_channels=3, use_checkpoint=True)


class UNet5b2i3o(UNet):
    """models.py:281-287"""

    def __init__(self):
        super().__init__(i_size=4, input_channels=2, out_channels=3, n_blocks=5, use_checkpoint=True)


class UNet4b1i3o(UNet):
    """models.py:290-296"""

    def __init__(self):
        super().__init__(i_size=7, input_channels=1, out_channels=3, use_checkpoint=True)


class UNetSP(UNet4b2i3o):
    """models.py:299-330 -- returns (encoded_full_skull, encoded_flap), each [B, 2, D, H, W]."""

    def __init__(self):
        super().__init__()
        self._head_mode = "sp"


class UNetSPSmall(UNet5b2i3o):
    """models.py:333-365 -- as UNetSP with a softmax over each encoded pair."""

    def __init__(self):
        super().__init__()
        self._head_mode = "sp_softmax"


class UNetDO(UNet4b1i3o):
    """models.py:368-387"""

    def __init__(self):
        super().__init__()
        self._head_mode = "sp"


# ---- legacy models (models.py:390-557) -------------------------------------------------------
def down_block_cr(in_c, out_c, kern_s, pad, dropout_p=0.5):
    """models.py:393-411"""
    return nn.Sequential(nn.Conv3d(in_c, out_c, kernel_size=kern_s, padding=pad),
                         nn.BatchNorm3d(out_c),
                         nn.ReLU(True),
                         nn.Conv3d(out_c, out_c, kernel_size=kern_s, padding=pad),
                         nn.BatchNorm3d(out_c),
                         nn.ReLU(True),
                         nn.Dropout3d(dropout_p))


def up_block_cr(in_c, out_c, kern_s_conv, kern_s_uconv, pad, stride_uc, dropout_p=0.5):
    """models.py:414-438"""
    return nn.Sequential(nn.ConvTranspose3d(in_c, in_c, kernel_size=kern_s_uconv, stride=stride_uc),
                         nn.Conv3d(in_c, out_c, kernel_size=kern_s_conv, padding=pad),
                         nn.BatchNorm3d(out_c),
                         nn.ReLU(True),
                         nn.Conv3d(out_c, out_c, kernel_size=kern_s_conv, padding=pad),
                         nn.BatchNorm3d(out_c),
                         nn.ReLU(True),
                         nn.Dropout3d(dropout_p))


class recAE_v2_fixed(_FusedNet):
    """models.py:441-538 -- 4 encoding/decoding blocks, 5^3 convolutions with bias, live center block,
    softmax head."""

    def __init__(self, input_channels=1, kern_sz_conv=5, kern_sz_upconv=2, stride_upconv=2, i_size=8, padding=2,
                 dropout_p=0, use_checkpoint=True):
        super().__init__()
        self.chk = use_checkpoint
        self.compute_dtype = _COMPUTE_DTYPE
        if kern_sz_upconv != 2 or stride_upconv != 2:
            raise NotImplementedError("the fused path covers ConvTranspose3d kernel 2 / stride 2 only")
        _check_conv_geometry(kern_sz_conv, padding)
        self._k = kern_sz_conv
        self._dropout_p = dropout_p
        self._dropout_rng = {}        # device -> engine.DropoutRNG (created by the first pass that draws masks there)
        fms = [i_size * pow(2, n) for n in range(5)]
        self.mp = nn.MaxPool3d(kernel_size=2, padding=0, stride=2, dilation=1, return_indices=True)
        self.dblock1 = down_block_cr(input_channels, fms[0], kern_s=kern_sz_conv, pad=padding, dropout_p=dropout_p)
        self.dblock2 = down_block_cr(fms[0], fms[1], kern_s=kern_sz_conv, pad=padding, dropout_p=dropout_p)
        self.dblock3 = down_block_cr(fms[1], fms[2], kern_s=kern_sz_conv, pad=padding, dropout_p=dropout_p)
        self.dblock4 = down_block_cr(fms[2], fms[3], kern_s=kern_sz_conv, pad=padding, dropout_p=dropout_p)
        self.cblock_center = nn.Sequential(nn.Conv3d(fms[3], fms[4], kernel_size=kern_sz_conv, padding=padding),
                                           nn.BatchNorm3d(fms[4]),
                                           nn.ReLU(True),
                                           nn.Conv3d(fms[4], fms[4], kernel_size=kern_sz_conv, padding=padding),
                                           nn.BatchNorm3d(fms[4]),
                                           nn.ReLU(True),
                                           nn.Dropout3d(dropout_p))
        self.ublock1 = up_block_cr(fms[4], fms[3], kern_sz_conv, kern_sz_upconv, padding, stride_upconv, dropout_p)
        self.ublock2 = up_block_cr(2 * fms[3], fms[2], kern_sz_conv, kern_sz_upconv, padding, stride_upconv, dropout_p)
        self.ublock3 = up_block_cr(2 * fms[2], fms[1], kern_sz_conv, kern_sz_upconv, padding, stride_upconv, dropout_p)
        self.ublock4 = up_block_cr(2 * fms[1], fms[0], kern_sz_conv, kern_sz_upconv, padding, stride_upconv, dropout_p)
        self.last_conv = nn.Conv3d(2 * fms[0], 2, kernel_size=1)

    def _levels(self):
        return 4

    def _dropout_sites(self):
        downs = [("dblock%d.6" % n, m[6], m[4].num_features)
                 for n, m in enumerate([self.dblock1, self.dblock2, self.dblock3, self.dblock4], 1)]
        ups = [("ublock%d.7" % n, m[7], m[5].num_features)
               for n, m in enumerate([self.ublock1, self.ublock2, self.ublock3, self.ublock4], 1)]
        return downs + [("cblock_center.6", self.cblock_center[6], self.cblock_center[4].num_features)] + ups

    def _run(self, eng: Engine, x, training):
        """recAE_v2_fixed.forward (models.py:509-538)."""
        k = self._k
        extra = 1 if self.chk else 0
        cur = eng.pack(x)
        eng.input_act = cur
        keep = self._draw_dropout(eng, x.shape[0])
        skips = []
        for i, seq in enumerate([self.dblock1, self.dblock2, self.dblock3, self.dblock4]):
            y = eng.conv([cur], seq[0].weight, seq[0].bias, k, [eng.want_input_grad if i == 0 else True], training,
                         leaf_input=(i == 0))
            a = eng.bn_relu(y, seq[1], training, extra)
            y = eng.conv([a], seq[3].weight, seq[3].bias, k, [True], training)
            s, cur = eng.bn_relu(y, seq[4], training, extra, pool=True, keep=keep.get("dblock%d.6" % (i + 1)))
            skips.append(s)
        seq = self.cblock_center
        y = eng.conv([cur], seq[0].weight, seq[0].bias, k, [True], training)
        a = eng.bn_relu(y, seq[1], training, extra)
        y = eng.conv([a], seq[3].weight, seq[3].bias, k, [True], training)
        cur = eng.bn_relu(y, seq[4], training, extra, keep=keep.get("cblock_center.6"))
        srcs = [cur]
        for i, seq in enumerate([self.ublock1, self.ublock2, self.ublock3, self.ublock4]):
            y = _up_stage(eng, srcs, seq[0], seq[1], k, training)
            a = eng.bn_relu(y, seq[2], training, extra)
            y = eng.conv([a], seq[4].weight, seq[4].bias, k, [True], training)
            up = eng.bn_relu(y, seq[5], training, extra, keep=keep.get("ublock%d.7" % (i + 1)))
            srcs = [up, skips[3 - i]]                                            # models.py:528-534
        return eng.head(srcs, self.last_conv.weight, self.last_conv.bias, _lib.HEAD_SOFTMAX)   # models.py:538


class UNet4_2IC(recAE_v2_fixed):
    """models.py:541-557"""

    def __init__(self):
        super().__init__(i_size=7, input_channels=2)
