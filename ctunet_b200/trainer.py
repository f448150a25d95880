"""The reference's step driver on the B200 path: one training / validation / test iteration.

Restates ``Model.forward_pass`` (ctunet/pytorch/Model.py:324-380) with the optimizers and the scheduler of
``Model.initialize_optimizer`` (Model.py:510-546):

  'train'   H2D copy, ``input.requires_grad_()``, forward, ``comp_losses_metrics``, ``backward``, ``optimizer.step()``,
            ``scheduler.step(loss)`` (ReduceLROnPlateau, every ITERATION, Model.py:369-371), ``param.grad = None``
            -> ``TrainStep``
  'val'     ``eval()``, no grad, forward, ``comp_losses_metrics`` (losses + Dice / Hausdorff metrics)    -> ``EvalStep``
  'test'    ``eval()``, no grad, forward, ``write_predictions`` = ``hard_segm_from_tensor`` per output + file IO
            (ProblemHandler.py:311-354)                                                                 -> ``EvalStep.labels``

The reference reads every loss component back with ``float(...)`` (five host syncs per batch, ProblemHandler.py:253-302)
and steps its scheduler on the host.  Here an iteration is a fixed sequence of launches of THIS library's kernels only --
the engine's tape (no autograd graph), the fused Dice+CE kernels, one loss-combine thread, one optimizer launch over all
parameters, one scheduler thread -- with no host synchronisation, so ``graph=True`` captures it ONCE in a CUDA graph
(after ``GRAPH_WARMUP`` eager iterations) and every later call is a copy of the batch into the graph's static inputs plus
one ``cudaGraphLaunch``.  The caller decides when to read the returned device tensor (``LossReadback``).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from . import engine as E
from ._lib import call, ptr_array, stream_ptr
from .engine import Engine
from .models import _run_planned
from .optim import FlatOptimizer
from .parallel import GradSync, PeerGradSync

# The head and the Dice + CrossEntropy loss as ONE pass over the head's inputs (forward) and one more (backward); off = the
# separate head / loss kernels the drop-in modules use behind the reference's model / handler split.
FUSED_HEAD_LOSS = True
GRAPH_WARMUP = 2      # eager iterations before the capture (allocator pools, cached constants, weight-preparation plan)


def _pair_fwd(pred, target, softmax_for_dice, want_ce):
    """ctu_dice_ce_fwd on one prediction / one-hot target pair -> (device float[2] = (CE mean, Dice loss), saved state)."""
    if pred.shape != target.shape or pred.dtype != torch.float32 or target.dtype != torch.float32:
        raise TypeError("prediction %s / target %s: float32 tensors of one [B, C, ...] shape expected"
                        % (tuple(pred.shape), tuple(target.shape)))
    pred, target = pred.contiguous(), target.contiguous()
    b, c = pred.shape[0], pred.shape[1]
    spatial = pred[0, 0].numel()
    sums = torch.empty(4 * b, dtype=torch.float64, device=pred.device)
    out = torch.empty(2, dtype=torch.float32, device=pred.device)
    call("ctu_dice_ce_fwd", pred.data_ptr(), target.data_ptr(), b, c, spatial, int(softmax_for_dice), int(want_ce),
         sums.data_ptr(), out.data_ptr(), stream_ptr())
    return out, (pred, target, sums, b, c, spatial, int(softmax_for_dice), int(want_ce))


def _pair_bwd(saved, g):
    pred, target, sums, b, c, spatial, sm, ce = saved
    dpred = torch.empty_like(pred)
    call("ctu_dice_ce_bwd", pred.data_ptr(), target.data_ptr(), b, c, spatial, sm, ce, sums.data_ptr(), g.data_ptr(),
         dpred.data_ptr(), stream_ptr())
    return dpred


class _LossSpec:
    """Which terms ``comp_losses_metrics`` sums, in the reference's order (ProblemHandler.py:59-91 / 241-298)."""

    def __init__(self, handler: str, dice_lambda: float, ce_lambda: float):
        if handler not in ("double", "single"):
            raise ValueError("handler: 'double' (FlapRecWithShapePriorDoubleOut) or 'single' (ProblemHandler)")
        self.handler = handler
        self.dice_lambda, self.ce_lambda = float(dice_lambda), float(ce_lambda)
        self.ce_on, self.dice_on = self.ce_lambda != 0, self.dice_lambda != 0
        if not (self.ce_on or self.dice_on):
            raise ValueError("both loss weights are zero")
        pairs = ("sk", "fl") if handler == "double" else ("",)
        self.keys = []
        if self.ce_on:
            self.keys += ["ce_" + p if p else "ce" for p in pairs]
        if self.dice_on:
            self.keys += ["dice_loss_" + p if p else "dice_loss" for p in pairs]
        self.keys.append("epoch_loss")
        self.n_terms = len(self.keys) - 1

    def forward(self, out, target, comps, mirror=None):
        """Enqueue the loss; fills ``comps`` (float[n_terms + 1], last = total).  Returns the saved state per pair."""
        if self.handler == "double":                          # softmax for the Dice term: ProblemHandler.py:233-235
            preds, tgts, sm = list(out), list(target), True
        else:
            preds, tgts, sm = [out], [target], False
        res = [_pair_fwd(p, t, sm, self.ce_on) for p, t in zip(preds, tgts)]
        terms, lams = [], []
        if self.ce_on:
            terms += [r[0][0:1] for r in res]
            lams += [self.ce_lambda] * len(res)
        if self.dice_on:
            terms += [r[0][1:2] for r in res]
            lams += [self.dice_lambda] * len(res)
        call("ctu_loss_combine", ptr_array([t.data_ptr() for t in terms]), (_lib.c_float * len(lams))(*lams), len(terms),
             comps.data_ptr(), mirror.data_ptr() if mirror is not None else None, stream_ptr())
        return [r[1] for r in res], [r[0] for r in res]


def _dropout_ps(model):
    """p of every Dropout3d site (a training step puts them all in train mode): what a captured step's masks depend on."""
    return tuple(float(m.p) for _, m, _ in model._dropout_sites())


class TrainStep:
    """``step(image, target)`` enqueues one full training iteration and returns the device tensor
    ``[components..., total]`` in the order of ``keys`` (no host sync).  In graph mode the returned tensor is the graph's
    static output: read it (or hand it to ``LossReadback``) before the next call.

    ``optimizer``: 'adam' | 'adamw' (amsgrad=True) | 'rmsprop' | 'sgd' with the reference's arguments (Model.py:514-541);
    ``scheduler=True`` (or a dict of ReduceLROnPlateau arguments): ``ReduceLROnPlateau()`` stepped after every iteration on that iteration's total loss (Model.py:369-371,
    544-546).  Data parallel: pass ``grad_sync=GradSync(model, ...)``; the loss every rank logs and feeds the scheduler is
    the mean over ranks (what the reference computes on the gathered batch).

    ``augment=utilities.RandomAffine(...)``: ``step_from_masks`` / ``step_from_bits`` draw one random affine transform per
    sample and encode the transformed masks straight into the step's inputs (``ctu_affine_encode_flaprec``; the atlas
    channel stays as it is), outside the captured graph like the plain encoders; ``last_affine()`` returns what the latest
    step drew.  Such a step takes masks only: ``__call__`` with a ready image raises ``ValueError``.

    ``craniectomy=utilities.RandomCraniectomy(...)``: the step takes the FULL skulls only (``step_from_skulls`` /
    ``step_from_skull_bits``) and cuts one random hole per sample on the device, fused into the same encoder launch (and
    with ``augment`` into the same gather: the hole is cut in skull space, then transformed); ``last_craniectomy()``
    returns the drawn holes.  ``__call__``, ``step_from_masks`` and ``step_from_bits`` take masks that are already cut and
    raise ``ValueError`` on such a step."""

    def __init__(self, model, handler: str = "double", dice_lambda: float = 1.0, ce_lambda: float = 1.0,
                 lr: float = 1e-4, weight_decay: float = 0.0, optimizer: str = "adam", momentum: float = 0.99,
                 scheduler=False, grad_sync: Optional[GradSync] = None, input_requires_grad: bool = True,
                 graph: bool = False, split_graph: Optional[bool] = None, augment=None, craniectomy=None):
        from .utilities import RandomAffine, RandomCraniectomy
        if augment is not None and not isinstance(augment, RandomAffine):
            raise TypeError("augment: a utilities.RandomAffine or None")
        if craniectomy is not None and not isinstance(craniectomy, RandomCraniectomy):
            raise TypeError("craniectomy: a utilities.RandomCraniectomy or None")
        self.model = model
        self.augment = augment
        self.craniectomy = craniectomy
        self._last_affine = None                              # (params, matrices) of the latest augmenting step
        self._last_craniectomy = None                         # params [B, 7] of the latest craniectomy step
        self.spec = _LossSpec(handler, dice_lambda, ce_lambda)
        self.handler, self.keys = handler, self.spec.keys
        self.input_requires_grad = input_requires_grad       # Model.py:351-352
        self.grad_sync = grad_sync
        # gradients always land in ONE flat buffer: the optimizer is a single launch over it, data parallel or not
        self.grads = grad_sync if grad_sync is not None else GradSync(model, deferred=True)
        self.world = self.grads.world
        # gradient exchange inside the optimizer kernel over NVLink peer memory: no collective call in the step
        self.peer = isinstance(self.grads, PeerGradSync)
        dev = self.grads.flat.device
        if not self.grads.flat.is_cuda:
            raise RuntimeError("TrainStep runs on CUDA only (no CPU fallback): move the model to the GPU first")
        if optimizer not in ("adam", "adamw", "rmsprop", "sgd"):
            raise ValueError("optimizer %r" % optimizer)
        self.optimizer = FlatOptimizer(self.grads.params, self.grads.flat, kind=optimizer, lr=lr, weight_decay=weight_decay,
                                       momentum=momentum if optimizer in ("rmsprop", "sgd") else 0.0, amsgrad=True,
                                       plateau=bool(scheduler), plateau_cfg=scheduler if isinstance(scheduler, dict) else None)
        self._g = torch.tensor([self.spec.ce_lambda, self.spec.dice_lambda], dtype=torch.float32, device=dev)
        self._comps = torch.zeros(self.spec.n_terms + 1, dtype=torch.float32, device=dev)
        self.graph = bool(graph)
        # two captured graphs around one eager all-reduce (data parallel), or one graph for the whole iteration
        self.split_graph = (self.world > 1 and not self.peer) if split_graph is None else bool(split_graph)
        self._graph = None
        self._graph_opt = None
        self._static = None
        self._static_out = None
        self._calls = 0
        self._dropout_cfg = None                              # Dropout3d sites / p the captured step draws masks for
        self.launches_per_step = None                         # C-ABI calls recorded in the captured step

    # ------------------------------------------------------------------ one iteration, enqueued on the current stream
    def _forward_backward(self, image: torch.Tensor, target):
        net = self.model
        net.train()
        net._validate(image)
        params = net._weight_tensors()
        eng = Engine(image.device, net.compute_dtype, record=True)
        eng.grad_sink = self.grads
        eng.want_input_grad = bool(self.input_requires_grad)
        mirror = self.grads.tail if (self.world > 1 or self.peer) else None
        if self.peer:
            self.grads.wait_released()                        # the flat buffer (loss tail first) is about to be rewritten
        if FUSED_HEAD_LOSS:
            # the head runs fused with the loss: the fp32 network outputs and their gradients are never materialised
            eng.fused_loss = (target, self.handler == "double", self.spec.ce_lambda, self.spec.dice_lambda, self._comps, mirror)
            _run_planned(net, eng, image.contiguous(), True, params)
            eng.backward()
        else:
            out = _run_planned(net, eng, image.contiguous(), True, params)
            saved, _ = self.spec.forward(out, target, self._comps, mirror)
            dpreds = [_pair_bwd(s, self._g) for s in saved]
            eng.backward(dpreds[0], dpreds[1] if len(dpreds) > 1 else None)
        self.grads.check_complete()
        if self.peer:
            self.grads.signal()
            return self.grads.tail_avg[:self.spec.n_terms + 1]       # filled by the fused exchange + optimizer kernel
        # world > 1: the averaged components come back in the tail of the flat buffer
        return self.grads.tail[:self.spec.n_terms + 1] if self.world > 1 else self._comps

    def _update(self, comps):
        if self.peer:
            self.optimizer.step_peer(self.grads, self.spec.n_terms + 1)
        else:
            self.optimizer.step(loss=comps[self.spec.n_terms:self.spec.n_terms + 1])

    def _eager(self, image, target):
        comps = self._forward_backward(image, target)
        self.grads.finish(publish=False)                      # data parallel: wait for / run the all-reduce
        self._update(comps)
        return comps

    def _no_craniectomy(self, what):
        if self.craniectomy is not None:
            raise ValueError("%s takes masks that are already cut: a TrainStep with craniectomy takes the full skulls "
                             "through step_from_skulls / step_from_skull_bits" % what)

    def __call__(self, image: torch.Tensor, target):
        self._no_craniectomy("__call__")
        if self.augment is not None:
            raise ValueError("an augmenting TrainStep transforms masks: feed it through step_from_masks / step_from_bits")
        return self._step(image, target)

    def _step(self, image: torch.Tensor, target):
        if not self.graph:
            return self._eager(image, target)
        self._calls += 1
        if self._graph is None and self._calls <= GRAPH_WARMUP:
            return self._eager(image, target)
        flat = [image] + (list(target) if isinstance(target, (tuple, list)) else [target])
        if self._graph is None:
            self._static = [torch.empty_like(t) for t in flat]
        elif any(a.shape != b.shape or a.dtype != b.dtype for a, b in zip(flat, self._static)):
            raise RuntimeError("graph mode: the batch shape changed after the step was captured")
        elif _dropout_ps(self.model) != self._dropout_cfg:
            raise RuntimeError("graph mode: the Dropout3d configuration (p of a site) changed after the step was captured")
        for dst, src in zip(self._static, flat):
            if dst.data_ptr() != src.data_ptr():              # a pipeline may fill static_inputs() in place
                dst.copy_(src, non_blocking=True)
        if self._graph is None:
            st_img = self._static[0]
            st_tgt = tuple(self._static[1:]) if isinstance(target, (tuple, list)) else self._static[1]
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            l0 = _lib.launches
            if not self.split_graph:
                with torch.cuda.graph(g, stream=E.chain_stream(st_img.device)):   # records the launches; nothing executes here
                    self._static_out = self._forward_backward(st_img, st_tgt)
                    self.grads.begin_step()
                    self._update(self._static_out)
            else:
                # data parallel: graph 1 = forward + loss + backward (gradients and the loss tail land in the flat
                # buffer), ONE eager NCCL all-reduce of that buffer, graph 2 = optimizer + scheduler
                if not self.grads.deferred:
                    raise RuntimeError("graph mode needs GradSync(deferred=True)")
                with torch.cuda.graph(g, stream=E.chain_stream(st_img.device)):
                    self._static_out = self._forward_backward(st_img, st_tgt)
                self.grads.begin_step()
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2, pool=g.pool()):
                    self._update(self._static_out)
                self._graph_opt = g2
            self.launches_per_step = _lib.launches - l0
            self._dropout_cfg = _dropout_ps(self.model)
            self._graph = g
        return self._replay()

    def static_inputs(self):
        """(image, target) buffers the captured graph reads, or None before the capture: a data pipeline that writes
        the next batch straight into them (and passes them to ``__call__``) saves the per-step device copy."""
        if self._graph is None:
            return None
        tgt = tuple(self._static[1:]) if len(self._static) > 2 else self._static[1]
        return self._static[0], tgt

    def _replay(self):
        self._graph.replay()
        if self._graph_opt is not None:
            self.grads.reduce_all()
            self._graph_opt.replay()
        return self._static_out

    def step_from_masks(self, broken: torch.Tensor, full: torch.Tensor, flap: torch.Tensor, atlas=None):
        """One iteration from the uint8 masks of a batch ([B,D,H,W] each, on the device): the float image (+ atlas channel)
        of datasets.py:195-235 is produced by ``ctu_encode_flaprec_u8`` straight into the captured graph's static input,
        and the label masks ARE the targets -- the fused head + loss kernels read them as uint8 (``one_hot`` of a {0,1}
        label is [1 - m, m]), so a training loop ships 3 bytes per voxel over PCIe instead of 24 and the one-hot float
        targets (16 bytes per voxel, read twice per step) never exist.  Without the fused head + loss, or when the step was
        captured with float targets, the one-hot targets are encoded as well."""
        from .utilities import encode_flaprec_batch
        self._no_craniectomy("step_from_masks")
        if self.handler != "double":
            raise ValueError("step_from_masks feeds the double-output handler (full skull + flap targets)")
        masks = FUSED_HEAD_LOSS and (self._graph is None or self._static[1].dtype == torch.uint8)
        if self.augment is not None:
            if not masks:
                raise ValueError("an augmenting step feeds uint8 label masks to the fused head + loss kernels")
            return self._augmented(0, (broken, full, flap), tuple(broken.shape[1:]), atlas)
        if self._graph is not None:
            if masks:
                encode_flaprec_batch(broken, full, flap, atlas, out=(self._static[0], None))
                for dst, src in ((self._static[1], full), (self._static[2], flap)):
                    if dst.data_ptr() != src.data_ptr():
                        dst.copy_(src, non_blocking=True)
            else:
                encode_flaprec_batch(broken, full, flap, atlas, out=(self._static[0], (self._static[1], self._static[2])))
            return self._replay()
        if masks:
            image = torch.empty((broken.shape[0], 1 if atlas is None else 2) + tuple(broken.shape[1:]), dtype=torch.float32,
                                device=broken.device)
            encode_flaprec_batch(broken, full, flap, atlas, out=(image, None))
            return self._step(image, (full.contiguous(), flap.contiguous()))
        image, target = encode_flaprec_batch(broken, full, flap, atlas)
        return self._step(image, target)

    def step_from_bits(self, broken_bits: torch.Tensor, full_bits: torch.Tensor, flap_bits: torch.Tensor, vol_shape, atlas=None):
        """``step_from_masks`` for BIT-PACKED masks ([B, D*H*W/8] uint8 each on the device, ``utilities.pack_mask_bits``):
        3 bits per voxel over PCIe.  ``ctu_encode_flaprec_bits`` expands them straight into the captured step's static
        inputs -- the float image (+ atlas) and the two uint8 label masks the fused head + loss kernels read."""
        from .utilities import encode_flaprec_bits
        self._no_craniectomy("step_from_bits")
        if self.handler != "double" or not FUSED_HEAD_LOSS:
            raise ValueError("step_from_bits feeds the double-output handler through the fused head + loss kernels")
        if self.augment is not None:
            return self._augmented(1, (broken_bits, full_bits, flap_bits), tuple(vol_shape), atlas)
        if self._graph is not None:
            if self._static[1].dtype != torch.uint8:
                raise RuntimeError("the step was captured with float targets: capture it through step_from_bits / step_from_masks")
            encode_flaprec_bits(broken_bits, full_bits, flap_bits, vol_shape, atlas,
                                out=(self._static[0], (self._static[1], self._static[2])))
            return self._replay()
        image, masks = encode_flaprec_bits(broken_bits, full_bits, flap_bits, vol_shape, atlas)
        return self._step(image, masks)

    def step_from_skulls(self, full: torch.Tensor, atlas=None):
        """One iteration from the FULL skulls of a batch (uint8 / bool [B, D, H, W] on the device, non-zero is bone):
        ``craniectomy`` draws one hole per sample and the fused encoder writes the broken skull (+ atlas) image and the
        full / flap label masks straight into the step's inputs -- no host synchronisation, one mask per sample."""
        if self.craniectomy is None:
            raise ValueError("step_from_skulls needs TrainStep(craniectomy=RandomCraniectomy(...))")
        if self.handler != "double" or not FUSED_HEAD_LOSS:
            raise ValueError("step_from_skulls feeds the double-output handler through the fused head + loss kernels")
        if not isinstance(full, torch.Tensor):
            raise TypeError("full: a uint8 [B, D, H, W] tensor")
        return self._augmented(0, (full,), tuple(full.shape[1:]), atlas)

    def step_from_skull_bits(self, full_bits: torch.Tensor, vol_shape, atlas=None):
        """``step_from_skulls`` for BIT-PACKED full skulls ([B, D*H*W/8] uint8 on the device, ``utilities.pack_mask_bits``):
        1 bit per voxel over PCIe."""
        if self.craniectomy is None:
            raise ValueError("step_from_skull_bits needs TrainStep(craniectomy=RandomCraniectomy(...))")
        if self.handler != "double" or not FUSED_HEAD_LOSS:
            raise ValueError("step_from_skull_bits feeds the double-output handler through the fused head + loss kernels")
        return self._augmented(1, (full_bits,), tuple(vol_shape), atlas)

    def _augmented(self, bits: int, srcs, vol, atlas):
        """Draw the batch's transforms and / or holes and encode the resulting masks into the step's inputs (the captured
        graph's static inputs once it exists): float image (+ the atlas, untransformed) and the two uint8 label masks.
        ``srcs``: the (broken, full, flap) masks, or with ``craniectomy`` the full skulls alone."""
        broken = srcs[0]
        what = ("one uint8 bit-packed [B, D*H*W/8] skull batch" if len(srcs) == 1 else
                "three uint8 bit-packed [B, D*H*W/8] masks of one shape") if bits else \
            ("one uint8 / bool [B, D, H, W] skull batch" if len(srcs) == 1 else "three uint8 [B, D, H, W] masks of one shape")
        for t in srcs:
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise RuntimeError("the masks must be CUDA tensors (no CPU fallback)")
            if t.dtype not in ((torch.uint8,) if bits else (torch.uint8, torch.bool)) or t.shape != broken.shape:
                raise TypeError("%s expected" % what)
        if len(vol) != 3:
            raise ValueError("vol_shape: (D, H, W)")
        b = broken.shape[0]
        d, h, w = (int(v) for v in vol)
        if (broken.dim() != 2 or broken.shape[1] * 8 != d * h * w) if bits else (broken.dim() != 4 or tuple(broken.shape[1:]) != vol):
            raise ValueError("masks %s do not match the volume shape %s" % (tuple(broken.shape), vol))
        cin = 1 if atlas is None else 2
        if atlas is not None and (atlas.dtype != torch.float32 or tuple(atlas.shape) != (d, h, w) or not atlas.is_cuda):
            raise TypeError("atlas: float32 CUDA volume of the mask shape")
        if self._graph is not None:
            if self._static[1].dtype != torch.uint8:
                raise ValueError("the step was captured with float targets: an augmenting step needs uint8 label masks")
            image, fm, lm = self._static
            if tuple(image.shape) != (b, cin, d, h, w):
                raise RuntimeError("graph mode: the batch shape changed after the step was captured")
        else:
            image = torch.empty((b, cin, d, h, w), dtype=torch.float32, device=broken.device)
            fm = torch.empty((b, d, h, w), dtype=torch.uint8, device=broken.device)
            lm = torch.empty_like(fm)
        src = [t.contiguous() for t in srcs]
        hole = None
        if self.craniectomy is not None:
            hole = self.craniectomy.draw(src[0], (d, h, w) if bits else None)
        mats = None
        if self.augment is not None:
            params, mats = self.augment.draw(b, (d, h, w), broken.device)
            self._last_affine = (params, mats)
        atlas_ptr = atlas.contiguous().data_ptr() if atlas is not None else None
        if hole is not None:
            call("ctu_craniectomy_encode_flaprec", bits, src[0].data_ptr(), hole.data_ptr(), atlas_ptr,
                 mats.data_ptr() if mats is not None else None, image.data_ptr(), fm.data_ptr(), lm.data_ptr(), b, cin, d, h,
                 w, stream_ptr())
            self._last_craniectomy = hole
        else:
            call("ctu_affine_encode_flaprec", bits, *[t.data_ptr() for t in src], atlas_ptr, mats.data_ptr(), image.data_ptr(),
                 fm.data_ptr(), lm.data_ptr(), b, cin, d, h, w, stream_ptr())
        if self._graph is not None:
            return self._replay()
        return self._step(image, (fm, lm))

    def last_affine(self):
        """``(params [B, 10], matrices [B, 3, 4])`` the latest augmenting step drew (``RandomAffine.draw``), or None; valid
        until the next step."""
        return self._last_affine

    def last_craniectomy(self):
        """params [B, 7] of the holes the latest craniectomy step drew (``RandomCraniectomy.draw``), or None."""
        return self._last_craniectomy

    @property
    def lr(self) -> float:
        return self.optimizer.lr


class EvalStep:
    """The 'val' / 'test' branches of ``Model.forward_pass`` (Model.py:334-337, 360-364, 376-380): eval-mode forward without
    gradients, then either the loss components (+ the Dice / Hausdorff metrics of ProblemHandler.py:277-295 when
    ``metrics=True``) or the hard labels ``write_predictions`` saves (``hard_segm_from_tensor`` per output,
    ProblemHandler.py:338-343).  ``graph=True`` captures each of the two per batch shape."""

    def __init__(self, model, handler: str = "double", dice_lambda: float = 1.0, ce_lambda: float = 1.0,
                 metrics: bool = False, graph: bool = False):
        self.model = model
        self.spec = _LossSpec(handler, dice_lambda, ce_lambda)
        self.handler = handler
        self.metrics = bool(metrics)
        self.keys = list(self.spec.keys[:-1])
        if self.metrics:
            sfx = ("_sk", "_fl") if handler == "double" else ("",)
            self.keys += ["dice_coef" + s for s in sfx]
            if handler == "double":                           # the base handler has no Hausdorff metric
                self.keys += ["hd_coef" + s for s in sfx]
        self.keys.append("epoch_loss")
        self.graph = bool(graph)
        self._captured = {}

    @torch.no_grad()
    def _forward(self, image):
        net = self.model
        was = net.training
        net.eval()
        try:
            return net(image)
        finally:
            net.train(was)

    def _validate_impl(self, image, target):
        from .utilities import dice_coeff, hausdorff
        out = self._forward(image)
        n = self.spec.n_terms
        comps = torch.empty(n + 1, dtype=torch.float32, device=image.device)
        self.spec.forward(out, target, comps)
        vals = [comps[:n]]
        if self.metrics:
            pairs = list(zip(out, target)) if self.handler == "double" else [(out, target)]
            vals.append(torch.stack([dice_coeff(p, t) for p, t in pairs]))
            if self.handler == "double":
                vals.append(torch.stack([hausdorff(p, t) for p, t in pairs]).float())
        vals.append(comps[n:])
        return torch.cat(vals)

    def _labels_impl(self, image):
        # the head kernel writes the hard labels itself (no fp32 outputs, no separate argmax pass)
        return self.model.predict_labels(image)

    def _run(self, which, fn, tensors):
        if not self.graph:
            return fn(*tensors)
        flat = []
        for t in tensors:
            flat += list(t) if isinstance(t, (tuple, list)) else [t]
        key = (which,) + tuple((tuple(t.shape), t.dtype) for t in flat)
        ent = self._captured.get(key)
        if ent is None:
            static = [torch.empty_like(t) for t in flat]
            for d, s in zip(static, flat):
                d.copy_(s)
            it = iter(static)
            args = [tuple(next(it) for _ in t) if isinstance(t, (tuple, list)) else next(it) for t in tensors]
            fn(*args)                                         # warm-up: weight-preparation plan, allocator pools
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                res = fn(*args)
            ent = (g, static, res)
            self._captured[key] = ent
        g, static, res = ent
        for d, s in zip(static, flat):
            d.copy_(s, non_blocking=True)
        g.replay()
        return res

    def __call__(self, image, target):
        """Device tensor of the values named by ``keys`` for one validation batch (no host sync)."""
        return self._run("val", self._validate_impl, (image, target))

    def labels(self, image):
        """Tuple of float32 label volumes [B, D, H, W], one per model output."""
        return self._run("test", self._labels_impl, (image,))


class LossReadback:
    """Deferred read-back of the loss components (SURVEY.md section 8f, rank 1).

    The reference reads every component with ``float(...)`` as soon as it exists (ProblemHandler.py:253-302): five host
    syncs per batch, each idling the GPU until the host has enqueued the next kernels.  Here every step's component
    tensor is copied asynchronously into pinned host memory on the step's stream; ``push`` returns the values of the
    PREVIOUS step (already complete, or waited for while the current step runs), ``drain`` the last one.  The
    ``losses_and_metrics`` lists (Model.py:363, ProblemHandler.py:71-102) receive the same floats, one step later."""

    def __init__(self, n_values: int, depth: int = 2):
        self.host = [torch.empty(n_values, dtype=torch.float32).pin_memory() for _ in range(depth)]
        self.events = [torch.cuda.Event() for _ in range(depth)]
        self.count = 0
        self.bytes_per_step = 4 * n_values

    def push(self, comps: torch.Tensor):
        slot = self.count % len(self.host)
        self.host[slot].copy_(comps, non_blocking=True)
        self.events[slot].record()
        self.count += 1
        lag = len(self.host) - 1                # depth 2: the previous step; depth 3: two steps back, ...
        return self._read(self.count - 1 - lag) if self.count > lag else None

    def drain(self):
        """Values of every step not yet returned by ``push`` (oldest first); the last entry is the final step's."""
        lag = len(self.host) - 1
        out = [self._read(i) for i in range(max(0, self.count - lag), self.count)]
        return out[-1] if out else None

    def _read(self, index: int):
        slot = index % len(self.host)
        self.events[slot].synchronize()
        return self.host[slot].tolist()
