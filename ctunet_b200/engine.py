"""Host-side executor of the U-Net hot path: a tape of fused stages over blocked activations.

Every stage is one or a few calls into the C ABI (include/ctunet_b200.h); PyTorch only owns the
memory and the stream.  A forward pass in training mode records a tape of backward closures; the
whole network is exposed to autograd as ONE ``torch.autograd.Function`` (see models.py), so a
training step is a fixed sequence of kernel launches with no host synchronisation and can be
captured in a CUDA graph.

Reference behaviour restated here (file:line relative to the reference root):
  * conv -> BatchNorm3d(train: batch statistics) -> ReLU stages   ctunet/pytorch/models.py:25-46
  * MaxPool3d(2,2) after every down block                           models.py:190-191, 233
  * channel concat of (up-block output, skip) folded into the consumer   models.py:249, 528-534
  * reentrant-checkpoint double update of BatchNorm running stats   models.py:232 (SURVEY App. D.2)
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence

import os

import torch

from . import _lib
from ._lib import CTU_ACCUM_PREZEROED, CTU_BF16, CTU_F32, call, int_array, ll_array, ptr_array, stream_ptr

BN_EPS = 1e-5
BN_FOLD_MAX_VOXELS = 4 * 64 ** 3      # see Engine.bn_relu

# "auto": tcgen05 implicit GEMM where the kernel covers the shape, CUDA-core direct kernel elsewhere;
# "direct": CUDA-core kernels only (always the case in fp32 accumulate-check mode).
CONV_PATH = "auto"

# "auto": ConvTranspose3d(k2,s2) + Conv3d of every up block run as ONE composed convolution on the low-resolution
# grid wherever the tcgen05 kernels cover it (bf16 mode); "off": never; "force": always (also in fp32 check mode,
# through the CUDA-core kernels -- used by the tests to check the composition at fp32 accuracy).
UP_FUSION = "auto"
_ONES = {}

# Re-pack all weights of a pass up front on a side stream (Engine.begin) instead of inline in the layer chain.
WEIGHT_PREP_ASYNC = True
# Weight gradients run on a second stream, overlapping the rest of the backward chain (Engine._conv_bwd).
WGRAD_ASYNC = True
# The discarded center block of the generic UNet runs on a third stream (Engine.off_critical_path).
DEAD_BRANCH_ASYNC = True
# The reduce pass of the BatchNorm+ReLU backward (sum dz, sum dz*xhat) folded into the epilogue of the data-gradient
# convolution that produces dA, when that convolution is the stage's only consumer and runs on the tcgen05 kernel.
# Correct (tests/test_gpu_upfuse.py) but OFF: measured on B200 it LOSES -- the epilogue is the bottleneck of the narrow
# convolutions, and the extra 16-byte load + 4 flops per element cost more there (six launches, +0.28 ms per step) than the
# separate bandwidth-bound reduce passes they replace (-0.2 ms): UNetSP step 4.40 -> 4.68 ms.
BN_BWD_FUSE = False
# The SP head's backward pass recovers the sigmoid values from the forward outputs instead of recomputing the logits.
HEAD_FROM_OUTPUTS = True
_SIDE = {}


# Stream priorities (captured into the graph's kernel nodes): the layer chain and the weight preparation it waits for run
# at HIGH priority, the leaves -- weight gradients, the dead center block, the network-input gradient -- at the default one.
# A leaf and the next link of the chain become runnable at the same moment (both wait for the same dy); without priorities
# the block scheduler took whichever was enqueued first, and a persistent weight-gradient kernel then held every SM (and its
# TMEM) for 100-250 us while the chain -- the critical path -- waited (CUPTI timeline, scripts/trace_step.py).
ACC_ARENA_DOUBLES = 32768   # 256 KB: every BatchNorm accumulator of a pass (forward sums + backward sums2)
# Weight images as batched index gathers (one launch per group of stages) instead of 2-4 packing launches per stage.
WEIGHT_GATHER = os.environ.get("CTU_WEIGHT_GATHER", "1") == "1"
_WEIGHT_MAPS: Dict[tuple, tuple] = {}     # layer signature -> (idx int32, count, bf16?)
STREAM_PRIORITIES = os.environ.get("CTU_PRIO", "1") == "1"
# When does the weight gradient of a stage join the race for the SMs?  A tcgen05 weight gradient and a tcgen05 data gradient
# cannot share an SM (TMEM), so whichever starts first makes the other wait.  Stages with ONE data gradient: weight gradient
# enqueued beside it (0).  Stages with two (the concatenated skip + up-sampled sources): behind them (2) -- otherwise it slips
# in between the two data gradients and the chain waits 150 us for it (CUPTI timeline; 4.254 -> 4.223 ms).  Always behind
# (1) is worse (4.32).  (A/B: CTU_WGRAD_AFTER=0/1/2)
# The ConvTranspose3d weight gradient (a CUDA-core kernel) stays IN the chain: beside it run the tcgen05 weight gradients of
# the stream next door, which it does not compete with for TMEM; moved onto that stream it queues behind them and the chain
# is left with data-gradient convolutions that do (measured: 4.30 -> 4.42 ms/step).  (A/B: CTU_CONVT_WGRAD_ASYNC=1)
# Leaf tails (gradient un-packing, weight-composition chain rule, BatchNorm buffer updates, head parameter gradients) on a
# third stream, and the weight-gradient accumulators pre-zeroed in arena chunks: the weight-gradient stream, which is the
# long pole of the backward pass, carries tcgen05 kernels only.  (A/B: CTU_LEAF_TAIL=0, CTU_WGRAD_ARENA=0)
LEAF_TAIL_ASYNC = os.environ.get("CTU_LEAF_TAIL", "1") == "1"
DEFER_BIG_WGRAD = os.environ.get("CTU_DEFER_WGRAD", "1") == "1"
DEFER_MIN_VOXELS = int(os.environ.get("CTU_DEFER_MIN_VOXELS", str(4 * 64 ** 3)))       # low-resolution voxels of the fused stage
DEFER_WINDOW_VOXELS = int(os.environ.get("CTU_DEFER_WINDOW_VOXELS", str(4 * 128 ** 3)))  # voxels x channel blocks of the BatchNorm
HEAD_PGRAD_LATE = int(os.environ.get("CTU_HEAD_PGRAD_LATE", "0"))   # 1: at the end of the tape; 2: beside the first data-gradient convolution    # (measured neutral to slightly negative: 4.25 vs 4.25-4.29 ms)
WGRAD_ARENA = os.environ.get("CTU_WGRAD_ARENA", "0") == "1"     # (measured: 4.274 with, 4.258 ms without -- the chunk memsets cost more than they save)
WACC_CHUNK_FLOATS = 4 * 1024 * 1024
CONVT_WGRAD_ASYNC = os.environ.get("CTU_CONVT_WGRAD_ASYNC", "0") == "1"
WGRAD_AFTER_DGRAD = int(os.environ.get("CTU_WGRAD_AFTER", "2"))      # 0 never, 1 always, 2 only for stages with >= 2 data gradients
_SIDE_HIGH = (0, 5)        # which: 0 weight preparation, 1 weight gradients, 2 dead branch, 3 network-input gradient,
                           # 4 leaf tails, 5 Dropout3d keep factors


def _side_stream(device, which=0):
    key = (str(device), which)
    if key not in _SIDE:
        prio = -1 if (STREAM_PRIORITIES and which in _SIDE_HIGH) else 0
        _SIDE[key] = torch.cuda.Stream(device=device, priority=prio)
    return _SIDE[key]


def chain_stream(device):
    """The high-priority stream a step is captured on (trainer.TrainStep / EvalStep graph mode)."""
    key = (str(device), "chain")
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device, priority=-1 if STREAM_PRIORITIES else 0)
    return _SIDE[key]


class Act:
    """A channel-blocked activation [N][Cb][D][H][W][8] (bf16 in product mode, fp32 in check mode).

    ``c_nat`` is set on the PHASE-MAJOR output of the fused up-sampling stage: the tensor then holds 8 phases x
    8*ceil(c_nat/8) channels on the low-resolution grid (block q*cb_nat + b), i.e. a [c_nat] x (2d, 2h, 2w) volume."""
    __slots__ = ("buf", "c", "n", "d", "h", "w", "sums", "c_nat", "bn")

    def __init__(self, buf, c, n, d, h, w):
        self.buf, self.c, self.n, self.d, self.h, self.w = buf, c, n, d, h, w
        self.sums = None        # per-channel sum / sum of squares written by the producing conv's epilogue
        self.c_nat = 0
        self.bn = None          # set on the output of a recorded BatchNorm+ReLU stage: see Engine.bn_relu (backward fusion)

    @property
    def cb(self):
        return (self.c + 7) // 8

    @property
    def spatial(self):
        return self.d * self.h * self.w

    @property
    def ptr(self):
        return self.buf.data_ptr()


_U64 = (1 << 64) - 1


def _splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & _U64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _U64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _U64
    return x ^ (x >> 31)


def philox_key(device, domain: int = 0) -> int:
    """64-bit Philox key of one random stream on ``device``: ``torch.initial_seed()`` mixed with the device index, the
    ``torch.distributed`` rank (when one is initialised) and ``domain``, a constant per consumer (0: Dropout3d) so that
    streams of different consumers never share a key."""
    device = torch.device(device)
    rank = 0
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        rank = torch.distributed.get_rank()
    idx = device.index if device.index is not None else torch.cuda.current_device()
    return _splitmix64(torch.initial_seed() ^ _splitmix64(((idx << 32) | (rank & 0xFFFFFFFF)) ^ domain))


class DropoutRNG:
    """Random state of the Dropout3d sites of one model on one device: a 64-bit Philox key and the pass counter, which
    lives in device memory and is advanced by the mask launch itself (ctu_dropout3d_keep), so a captured step draws new
    masks on every replay.  The key is ``torch.initial_seed()`` at creation (``torch.manual_seed(s)`` reproduces a run),
    mixed with the device index (``nn.DataParallel`` replicas) and the ``torch.distributed`` rank when one is initialised,
    so replicas and ranks draw independent masks."""
    __slots__ = ("key", "counter", "last")

    def __init__(self, device):
        self.key = philox_key(device)
        self.counter = torch.zeros(1, dtype=torch.int64, device=device)
        self.last = {}          # site name -> [N, C] view of the keep factors of the last pass that drew masks


class Engine:
    def __init__(self, device, compute_dtype: str, record: bool):
        if compute_dtype not in ("bf16", "fp32"):
            raise ValueError("compute dtype must be 'bf16' or 'fp32'")
        _lib.load()
        self.device = device
        self.tdtype = torch.bfloat16 if compute_dtype == "bf16" else torch.float32
        self.dtype = CTU_BF16 if compute_dtype == "bf16" else CTU_F32
        self.record = record
        self.tape: List[Callable[[], None]] = []
        self.agrads: Dict[int, Act] = {}            # id(Act) -> gradient Act
        self.pgrads: Dict[int, torch.Tensor] = {}   # id(param) -> gradient tensor
        self.want_input_grad = False
        self.input_grad = None                      # NCDHW fp32 gradient of the network input (leaf_input convolution)
        self.grad_sink = None                       # parallel.GradSync: gradients land in its flat buffer
        self.use_tc = (CONV_PATH == "auto" and compute_dtype == "bf16" and bool(_lib.load().ctu_has_tensor_path()))
        # weight preparation plan (see begin()): None = not in use, every preparation runs inline
        self._plan = None
        self._recording = False
        self._results = []
        self._pi = 0
        self._side = None
        self._wgrad_stream = None
        self._input_grad_stream = None
        self._arena = None
        self._arena_used = 0
        self._gjobs = []                           # pending weight-image gathers (see _kernel_weights)
        self._wacc = {}                            # stream -> [zeroed fp32 arena chunk, floats used] (see wacc)
        self._leaf_tail_stream = None
        self._late_leaves = []
        self._deferred_wgrads = []
        self._dead_stream = None
        # set by trainer.TrainStep: (targets, softmax_for_dice, ce_lambda, dice_lambda, comps, mirror) -- the head then
        # runs fused with the loss (csrc/head.cu: head_loss_*), produces no output tensors and wires its own backward
        self.fused_loss = None
        # inference epilogue (models._FusedNet.predict_labels): (vol, origins, patch) replaces the input pack by a patch
        # gather, (labels, origins, patch, dims) makes the head write hard labels (scattered at the origins when given)
        self.patch_src = None
        self.label_dst = None
        # overlapping windows (models._FusedNet.accumulate_windows): (acc, origins, patch, dims, weight table) makes the
        # head add its weighted outputs to the int64 accumulators instead (csrc/head.cu: head_accum_kernel)
        self.accum_dst = None
        self._keep_event = None                    # Dropout3d keep factors drawn on their own stream (see dropout_masks)

    # ------------------------------------------------------------------ weight preparation on a side stream
    def begin(self, store: dict, key) -> None:
        """Weight re-packing (native fp32 -> packed -> bf16 UMMA image, data-gradient packs, the composed weights
        of the fused up stage) depends on the parameters only.  The first pass with a given ``key`` (input shape,
        mode, flags) runs those ~100 tiny kernels inline and records them; every later pass enqueues ALL of them up
        front on a side stream -- off the critical path of the layer chain (parallel branches of the CUDA graph) --
        and each consumer just waits for its event."""
        if not WEIGHT_PREP_ASYNC:
            return
        plan = store.get(key)
        if plan is None:
            self._plan, self._recording = [], True
            self._store, self._key = store, key
            return
        self._plan = plan
        main = torch.cuda.current_stream()
        side = _side_stream(self.device)
        self._side = side
        side.wait_stream(main)
        with torch.cuda.stream(side):
            # Weight images are index gathers collected by _kernel_weights and launched in batches (ctu_gather_batch): one
            # launch for every stage up to the next weight COMPOSITION (a real computation: the stages before it must not
            # wait for it), one more right behind it.  All results of a batch share its event.
            pending = []

            def flush():
                if not pending and not self._gjobs:
                    return
                self._flush_gathers()
                ev = torch.cuda.Event()
                ev.record(side)
                for slot in pending:
                    slot[2] = ev
                pending.clear()

            for tag, fn, heavy in plan:
                if heavy:
                    flush()
                out = fn(self)
                for t in out:
                    if isinstance(t, torch.Tensor):
                        t.record_stream(main)
                slot = [tag, out, None]
                self._results.append(slot)
                pending.append(slot)
                if heavy:
                    flush()
            flush()

    def end_forward(self) -> None:
        """Publish a freshly recorded plan / join the side streams (required before a graph capture ends)."""
        if self._recording:
            self._store[self._key] = self._plan
            self._recording = False
        elif self._side is not None:
            torch.cuda.current_stream().wait_stream(self._side)
        if self._dead_stream is not None:
            torch.cuda.current_stream().wait_stream(self._dead_stream)
            self._dead_stream = None
        self._wait_keep()                            # (masks nobody applied: still joined, e.g. for a graph capture)

    # ------------------------------------------------------------------ Dropout3d keep factors
    def dropout_masks(self, rng: DropoutRNG, n: int, sites):
        """Draw the keep factors of every active Dropout3d site of this pass in ONE launch on a side stream (they depend on
        nothing but the random state, so they are off the layer chain).  ``sites``: [(site id, channels, p)]; returns one
        float32 [n, cpad] tensor per site.  The first BatchNorm stage that applies them waits for the launch."""
        cpads = [(c + 7) // 8 * 8 for _, c, _ in sites]
        main = torch.cuda.current_stream()
        side = _side_stream(self.device, 5)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            buf = self.f32(n * sum(cpads))
            call("ctu_dropout3d_keep", len(sites), int_array([s[0] for s in sites]), int_array([s[1] for s in sites]),
                 (_lib.c_float * len(sites))(*[float(s[2]) for s in sites]), n, rng.key, rng.counter.data_ptr(),
                 buf.data_ptr(), stream_ptr())
            ev = torch.cuda.Event()
            ev.record(side)
        buf.record_stream(main)
        self._keep_event = ev
        out, off = [], 0
        for cp in cpads:
            out.append(buf[off:off + n * cp].view(n, cp))
            off += n * cp
        return out

    def _wait_keep(self):
        if self._keep_event is not None:
            torch.cuda.current_stream().wait_event(self._keep_event)
            self._keep_event = None

    def off_critical_path(self, *inputs: "Act"):
        """Context: run stages whose OUTPUT nobody consumes (the generic UNet's discarded center block,
        models.py:238-241 -- only its BatchNorm buffers matter) on their own stream, beside the decoder."""
        import contextlib
        if not DEAD_BRANCH_ASYNC:
            return contextlib.nullcontext()
        main = torch.cuda.current_stream()
        side = _side_stream(self.device, 2)
        side.wait_stream(main)
        for a in inputs:
            a.buf.record_stream(side)
        self._dead_stream = side
        return torch.cuda.stream(side)

    def _prepared(self, tag: str, fn, heavy: bool = False):
        """``fn(engine) -> tuple of tensors`` computed from parameters and static shapes only.  ``heavy``: the
        preparation launches real work (a weight composition), see begin_forward()."""
        if self._plan is None or self._recording:
            if self._recording:
                self._plan.append((tag, fn, heavy))
            out = fn(self)
            self._flush_gathers()               # inline use: the consumer is about to be enqueued on this stream
            return out
        if self._pi >= len(self._results) or self._results[self._pi][0] != tag:
            raise RuntimeError("internal: weight preparation plan out of step at %r" % tag)
        _, out, ev = self._results[self._pi]
        self._pi += 1
        torch.cuda.current_stream().wait_event(ev)
        return out

    # ------------------------------------------------------------------ helpers
    def new_act(self, c, n, d, h, w) -> Act:
        cb = (c + 7) // 8
        return Act(torch.empty((n, cb, d, h, w, 8), dtype=self.tdtype, device=self.device), c, n, d, h, w)

    def f32(self, *shape):
        return torch.empty(shape, dtype=torch.float32, device=self.device)

    def f64(self, *shape):
        return torch.empty(shape, dtype=torch.float64, device=self.device)

    def acc64(self, n: int) -> torch.Tensor:
        """A ZEROED float64 accumulator of ``n`` entries (BatchNorm sums): a slice of one arena zeroed once per pass, so
        the ~30 per-layer memset nodes leave the layer chain (``_pz`` tells the library not to enqueue its own)."""
        if self._arena is None:
            self._arena = torch.zeros(ACC_ARENA_DOUBLES, dtype=torch.float64, device=self.device)
            self._arena_used = 0
        n16 = (n + 15) // 16 * 16
        if self._arena_used + n16 > ACC_ARENA_DOUBLES:
            return self.f64(n)                       # (arena exhausted: an ordinary buffer, zeroed by the entry point)
        t = self._arena[self._arena_used:self._arena_used + n]
        self._arena_used += n16
        t._ctu_prezeroed = True
        return t

    def wacc(self, n: int) -> torch.Tensor:
        """A ZEROED float32 buffer of ``n`` entries for a weight-gradient kernel (it accumulates with atomics): slices of
        arena chunks zeroed once on the stream that uses them, instead of one memset node in front of every kernel."""
        if not WGRAD_ARENA:
            return self.f32(n)
        n64 = (n + 63) // 64 * 64
        if n64 > WACC_CHUNK_FLOATS:
            t = torch.zeros(n, dtype=torch.float32, device=self.device)
            t._ctu_prezeroed = True
            return t
        key = torch.cuda.current_stream().cuda_stream
        ent = self._wacc.get(key)
        if ent is None or ent[1] + n64 > WACC_CHUNK_FLOATS:
            ent = [torch.zeros(WACC_CHUNK_FLOATS, dtype=torch.float32, device=self.device), 0]
            self._wacc[key] = ent
        t = ent[0][ent[1]:ent[1] + n]
        ent[1] += n64
        t._ctu_prezeroed = True
        return t

    def _leaf_tail(self, after_stream, fn, *tensors):
        """Run ``fn`` (small kernels that finish a LEAF of the backward pass: gradient un-packing, the chain rule of a
        weight composition, parameter-gradient registration, BatchNorm buffer updates) on the leaf-tail stream once
        ``after_stream`` has reached this point -- the weight-gradient stream carries tcgen05 kernels only."""
        if not LEAF_TAIL_ASYNC:
            with torch.cuda.stream(after_stream):
                fn()
            return
        tail = _side_stream(self.device, 4)
        tail.wait_stream(after_stream)
        with torch.cuda.stream(tail):
            fn()
        for t in tensors:
            if isinstance(t, torch.Tensor):
                t.record_stream(tail)
        self._leaf_tail_stream = tail

    @staticmethod
    def _pz(t) -> int:
        return CTU_ACCUM_PREZEROED if (t is not None and getattr(t, "_ctu_prezeroed", False)) else 0

    def _grad_buffer(self, param) -> torch.Tensor:
        """Where a parameter-gradient kernel writes: a slice of the data-parallel flat buffer, or a new tensor."""
        if self.grad_sink is not None:
            buf = self.grad_sink.buffer_for(param)
            if buf is not None:
                return buf
        return torch.empty_like(param)

    def _add_pgrad(self, param, g):
        k = id(param)
        if k in self.pgrads:
            raise RuntimeError("internal: parameter received two gradients")
        self.pgrads[k] = g
        if self.grad_sink is not None:
            self.grad_sink.delivered(param)

    def _consume(self, srcs):
        """Count the consumers of BatchNorm+ReLU outputs (the backward fusion needs exactly one)."""
        if self.record:
            for s in srcs:
                if s.bn is not None:
                    s.bn["consumers"] += 1

    @staticmethod
    def _src_args(srcs: Sequence[Act]):
        return ptr_array([s.ptr for s in srcs]), int_array([s.c for s in srcs]), len(srcs)

    def _tc_ok(self, k, srcs, cout):
        """0 = CUDA-core kernel, 1 = conv_tc.cu (weights resident in shared memory), 2 = conv_wide.cu (weights streamed)."""
        s0 = srcs[0]
        return tc_variant(k, [s.c for s in srcs], cout, s0.n, s0.d, s0.h, s0.w) if self.use_tc else 0

    def _kernel_weights(self, native, cout, k, chans, tc, dgrad_of=None, dims=None):
        """Kernel-ready weights of conv(cat(srcs with ``chans`` channels)) -> cout: the packed fp32 tensor (CUDA-core
        kernel) or the bf16 UMMA image (tcgen05 kernel).  ``dgrad_of = (i, cs)``: instead the weights of the data
        gradient dy (cout channels) -> d(src i) (cs channels).

        Every variant is a fixed permutation + cast of ``native``: the permutation is computed once per signature
        (``_weight_index_map`` runs the packing kernels on index-valued inputs) and the result is produced by one job of a
        batched gather -- PENDING until ``_flush_gathers()`` (the callers in _prepared / begin_forward flush)."""
        if not WEIGHT_GATHER:
            return self._kernel_weights_chain(native, cout, k, chans, tc, dgrad_of, dims)
        key = (tuple(native.shape), cout, k, tuple(chans), int(tc), dgrad_of, tuple(dims) if (tc == 2 and dims) else None,
               str(self.device))
        ent = _WEIGHT_MAPS.get(key)
        if ent is None:
            if torch.cuda.is_current_stream_capturing():
                # (a capture without a preceding eager pass: the map construction must not become part of the graph)
                return self._kernel_weights_chain(native, cout, k, chans, tc, dgrad_of, dims)
            ent = self._weight_index_map(native, cout, k, chans, tc, dgrad_of, dims)
            torch.cuda.current_stream().synchronize()      # once per signature: complete before any stream reads it
            _WEIGHT_MAPS[key] = ent
        idx, count, is_bf16 = ent
        src = native if native.is_contiguous() else native.contiguous()
        dst = (torch.empty(count * 2, dtype=torch.uint8, device=self.device) if is_bf16
               else torch.empty(count, dtype=torch.float32, device=self.device))
        self._gjobs.append((src, dst, idx, count, is_bf16))
        return dst

    def _weight_index_map(self, native, cout, k, chans, tc, dgrad_of, dims):
        """(idx int32 [count], count, bf16?) with out[i] = native.flatten()[idx[i]] (idx < 0: a zero pad entry) for the chain
        of packing launches of ``_kernel_weights_chain``.  The chain's last stage rounds to bf16 (8 significant bits), so the
        1-based source index travels through it as three base-256 digits."""
        n = native.numel()
        if n >= (1 << 24):
            raise RuntimeError("weight tensor too large for the index-map construction (%d elements)" % n)
        ar = torch.arange(1, n + 1, dtype=torch.int64, device=self.device)
        total = None
        is_bf16 = bool(tc)
        for digit in range(3 if is_bf16 else 1):
            if is_bf16:
                src = ((ar >> (8 * digit)) & 255).to(torch.float32).view(native.shape)
            else:
                src = ar.to(torch.float32).view(native.shape)          # fp32 holds every index below 2^24 exactly
            out = self._kernel_weights_chain(src, cout, k, chans, tc, dgrad_of, dims)
            vals = (out.view(torch.bfloat16) if is_bf16 else out).to(torch.float32).round().to(torch.int64)
            total = vals << (8 * digit) if total is None else total + (vals << (8 * digit))
        idx = (total - 1).to(torch.int32).contiguous()
        count = idx.numel()
        if count % 8:
            raise RuntimeError("internal: weight image of %d entries is not a multiple of 8" % count)
        return idx, count, is_bf16

    def _flush_gathers(self):
        """Launch the pending weight gathers as one batch on the current stream."""
        jobs, self._gjobs = self._gjobs, []
        if not jobs:
            return
        cur = torch.cuda.current_stream()
        for src, dst, idx, _, _ in jobs:
            for t in (src, dst, idx):
                t.record_stream(cur)
        call("ctu_gather_batch", len(jobs), ptr_array([j[0].data_ptr() for j in jobs]), ptr_array([j[1].data_ptr() for j in jobs]),
             ptr_array([j[2].data_ptr() for j in jobs]), ll_array([j[3] for j in jobs]), int_array([int(j[4]) for j in jobs]),
             stream_ptr())

    def _kernel_weights_chain(self, native, cout, k, chans, tc, dgrad_of=None, dims=None):
        """The packing launches themselves (native -> packed fp32 -> bf16 image): the definition the index maps are taken from."""
        lib = _lib.load()
        ca, ns, st = int_array(chans), len(chans), stream_ptr()
        if dgrad_of is None:
            wp = self.f32(lib.ctu_conv_wpack_floats(cout, k, ns, ca))
            call("ctu_conv_pack_weight", native.data_ptr(), wp.data_ptr(), cout, k, ns, ca, st)
            kin, kout = (ns, ca), cout
        else:
            i, cs = dgrad_of
            wp = self.f32(lib.ctu_conv_wpack_dgrad_floats(cout, k, cs))
            call("ctu_conv_pack_weight_dgrad", native.data_ptr(), wp.data_ptr(), cout, k, ns, ca, i, st)
            kin, kout = (1, int_array([cout])), cs
        if not tc:
            return wp
        if tc == 2:      # weight-streaming kernel: the image depends on the launch geometry (dims = n, d, h, w)
            cin1 = kin[1][0]
            wimg = torch.empty(lib.ctu_conv_wide_wimg_bytes(k, cin1, kout, *dims), dtype=torch.uint8, device=self.device)
            call("ctu_conv_wide_pack_weight", wp.data_ptr(), wimg.data_ptr(), k, cin1, kout, *dims, st)
            return wimg
        wimg = torch.empty(lib.ctu_conv_tc_wimg_bytes(k, kin[0], kin[1], kout), dtype=torch.uint8, device=self.device)
        call("ctu_conv_tc_pack_weight", wp.data_ptr(), wimg.data_ptr(), k, kin[0], kin[1], kout, st)
        return wimg

    def _conv_launch(self, srcs, wk, tc, bias, y: Act, cout, k, sums, stat_cout=0):
        """One forward-style convolution launch (also used for the data gradient) with kernel-ready weights."""
        s0 = srcs[0]
        pa, ca, ns = self._src_args(srcs)
        call("ctu_conv3d_fprop", self.dtype, pa, ca, ns, wk.data_ptr(), bias.data_ptr() if bias is not None else None,
             y.ptr, sums.data_ptr() if sums is not None else None, stat_cout, cout, k, s0.n, s0.d, s0.h, s0.w,
             int(tc) | self._pz(sums), stream_ptr())

    # ------------------------------------------------------------------ layout
    def pack(self, x: torch.Tensor) -> Act:
        if self.patch_src is not None:
            vol, origins, patch = self.patch_src
            c, vd, vh, vw = vol.shape
            a = self.new_act(c, origins.shape[0], patch, patch, patch)
            call("ctu_pack_patches", vol.data_ptr(), origins.data_ptr(), a.ptr, self.dtype, origins.shape[0], c, vd, vh, vw, patch,
                 stream_ptr())
            return a
        n, c, d, h, w = x.shape
        a = self.new_act(c, n, d, h, w)
        call("ctu_pack_ncdhw", x.data_ptr(), a.ptr, self.dtype, n, c, d * h * w, stream_ptr())
        return a

    def unpack(self, a: Act) -> torch.Tensor:
        out = self.f32(a.n, a.c, a.d, a.h, a.w)
        call("ctu_unpack_ncdhw", a.ptr, out.data_ptr(), self.dtype, a.n, a.c, a.spatial, stream_ptr())
        return out

    # ------------------------------------------------------------------ Conv3d
    def _conv_weights(self, tag, srcs, need, w_native, k, cout, compose=None):
        """Prepared weights of one convolution stage: (forward weights, [data-gradient weights per source or None],
        extra).  ``compose(engine) -> (w_native, extra...)`` builds the native weights first (fused up stage)."""
        chans = [s.c for s in srcs]
        s0 = srcs[0]
        tc_f = self._tc_ok(k, srcs, cout)
        dims = (s0.n, s0.d, s0.h, s0.w)
        tc_d = [tc_variant(k, [cout], s.c, *dims) if (nd and self.use_tc) else 0 for s, nd in zip(srcs, need)]
        need = list(need)

        def prep(eng):
            extra = ()
            wn = w_native
            if compose is not None:
                res = compose(eng)
                wn, extra = res[0], tuple(res[1:])
            out = [eng._kernel_weights(wn, cout, k, chans, tc_f, dims=dims)]
            for i, nd in enumerate(need):
                out.append(eng._kernel_weights(wn, cout, k, chans, tc_d[i], (i, chans[i]), dims=dims) if nd else None)
            return tuple(out) + (wn,) + extra

        res = self._prepared(tag, prep, heavy=compose is not None)
        ns = len(srcs)
        return res[0], tc_f, list(res[1:1 + ns]), tc_d, res[1 + ns], res[2 + ns:]

    def _conv_fwd(self, srcs, wk, tc, bias, k, cout, stat_cout, bn_stats):
        """y = conv(cat(srcs)) (+bias) with kernel-ready weights; returns the output activation."""
        s0 = srcs[0]
        y = self.new_act(cout, s0.n, s0.d, s0.h, s0.w)
        if bn_stats:
            y.sums = self.acc64(2 * (((stat_cout or cout) + 7) // 8 * 8))
        self._conv_launch(srcs, wk, tc, bias, y, cout, k, y.sums, stat_cout)
        return y

    def _conv_bwd(self, srcs, need, wkd, tc_d, y, k, cout, dw_out, db_out, after_wgrad=None, phase_cout=0,
                  leaf_input=False):
        """Weight gradient into ``dw_out`` (native layout, nullable) / ``db_out`` and the data gradient of every
        source with ``need[i]`` (prepared weights ``wkd[i]``).

        The weight gradient is a leaf of the backward graph (only the optimizer reads it), so it is enqueued on a
        second stream (``WGRAD_ASYNC``): it overlaps the BatchNorm / head kernels of the layers below while the data
        gradient stays on the critical path.  The un-packing into the native layout and ``after_wgrad()`` (small, non-tensor
        kernels) run behind it on a THIRD stream (``_leaf_tail``), so the next tcgen05 weight gradient is not queued behind them."""
        lib = _lib.load()
        s0 = srcs[0]
        dy = self.agrads.pop(id(y))
        pa, ca, ns = self._src_args(srcs)
        if dw_out is not None:
            def wgrad_kernel():
                dwp = self.wacc(lib.ctu_conv_wpack_floats(cout, k, ns, ca))
                tc = wgrad_variant(k, [s.c for s in srcs], cout, s0.d, s0.h, s0.w, phase_cout) if self.use_tc else 0
                call("ctu_conv3d_wgrad", self.dtype, pa, ca, ns, dy.ptr, dwp.data_ptr(),
                     db_out.data_ptr() if db_out is not None else None, phase_cout, cout, k, s0.n, s0.d, s0.h, s0.w,
                     int(tc) | self._pz(dwp), stream_ptr())
                return dwp

            def wgrad_tail(dwp):
                call("ctu_conv_unpack_wgrad", dwp.data_ptr(), dw_out.data_ptr(), cout, k, ns, ca, stream_ptr())
                if after_wgrad is not None:
                    after_wgrad()

        def enqueue_wgrad():
            main = torch.cuda.current_stream()
            side = _side_stream(self.device, 1)
            side.wait_stream(main)                      # dy (and everything enqueued before this point) is ready
            with torch.cuda.stream(side):
                dwp = wgrad_kernel()
            dy.buf.record_stream(side)
            self._wgrad_stream = side
            self._leaf_tail(side, lambda: wgrad_tail(dwp), dwp)

        def launch_wgrad():
            if dw_out is None:
                return
            if WGRAD_ASYNC:
                # The long weight gradients of the fused up stages at the top levels are held back until the chain reaches
                # a long BatchNorm-backward window (see _release_deferred_wgrad): tensor work under non-tensor work.
                if DEFER_BIG_WGRAD and phase_cout and s0.n * s0.d * s0.h * s0.w >= DEFER_MIN_VOXELS:
                    self._deferred_wgrads.append(enqueue_wgrad)
                else:
                    enqueue_wgrad()
            else:
                wgrad_tail(wgrad_kernel())

        after = WGRAD_AFTER_DGRAD == 1 or (WGRAD_AFTER_DGRAD == 2 and sum(1 for nd in need if nd) >= 2)
        if not after:
            launch_wgrad()

        def dgrads():
            if HEAD_PGRAD_LATE == 2 and self._late_leaves and any(need):
                for fn, keep in self._late_leaves:          # (CUDA-core leaves beside a tensor kernel, not beside BatchNorm)
                    self._leaf_tail(torch.cuda.current_stream(), fn, keep)
                self._late_leaves = []
            for i, s in enumerate(srcs):
                if not need[i]:
                    continue
                dx = self.new_act(s.c, s.n, s.d, s.h, s.w)
                info = s.bn
                if (BN_BWD_FUSE and info is not None and info["consumers"] == 1 and not info["pool"] and tc_d[i] == 1
                        and self.dtype == CTU_BF16 and not info["drop"]
                        and lib.ctu_conv_tc_bnred_supported(k, 1, int_array([cout]), s.c, s.d, s.h, s.w)):
                    # dx is dA of a BatchNorm+ReLU stage consumed only here: its backward reductions ride in this epilogue
                    sums2 = self.f64(2 * ((s.c + 7) // 8 * 8))
                    call("ctu_conv3d_dgrad_bnred", ptr_array([dy.ptr]), int_array([cout]), 1, wkd[i].data_ptr(), dx.ptr, s.c, k,
                         s.n, s.d, s.h, s.w, info["y"].ptr, info["ss"].data_ptr(), sums2.data_ptr(), info["pm"], stream_ptr())
                    info["sums2"] = sums2
                else:
                    self._conv_launch([dy], wkd[i], tc_d[i], None, dx, s.c, k, None)
                self._set_agrad(s, dx)

        if leaf_input and WGRAD_ASYNC and any(need):
            # The gradient of the NETWORK INPUT (the reference asks for it only because reentrant checkpointing needs an
            # input that requires grad, Model.py:351-352; nothing consumes it): a leaf like the weight gradients, so it is
            # computed and converted to NCDHW on the second stream, off the critical path; run_tape() joins that stream.
            main = torch.cuda.current_stream()
            side = _side_stream(self.device, 3)        # its own stream: beside the first layer's weight gradient, not behind it
            side.wait_stream(main)
            with torch.cuda.stream(side):
                dgrads()
                self.input_grad = self.unpack(self.agrads.pop(id(srcs[0])))
            self.input_grad.record_stream(main)
            dy.buf.record_stream(side)
            self._input_grad_stream = side
        else:
            dgrads()
        if after:
            launch_wgrad()

    def _pgrad_done(self, pairs):
        """Register parameter gradients produced on the current stream (see _add_pgrad)."""
        for prm, g in pairs:
            if g is not None:
                self._add_pgrad(prm, g)

    def conv(self, srcs: Sequence[Act], weight, bias, k: int, need_src_grad: Sequence[bool],
             bn_stats: bool = False, leaf_input: bool = False) -> Act:
        """``bn_stats``: also produce the batch statistics of the output (``y.sums``) for the BatchNorm that follows.
        ``leaf_input``: ``srcs[0]`` is the network input (its gradient is a leaf of the backward pass)."""
        cout = weight.shape[0]
        srcs = list(srcs)
        self._consume(srcs)
        need = [bool(n) and self.record for n in need_src_grad]
        wk, tc, wkd, tc_d, _, _ = self._conv_weights("conv", srcs, need, weight, k, cout)
        y = self._conv_fwd(srcs, wk, tc, bias, k, cout, 0, bn_stats)
        if self.record:
            def bwd():
                dw = self._grad_buffer(weight) if weight.requires_grad else None
                db = self._grad_buffer(bias) if (dw is not None and bias is not None and bias.requires_grad) else None
                self._conv_bwd(srcs, need, wkd, tc_d, y, k, cout, dw, db,
                               lambda: self._pgrad_done(((weight, dw), (bias, db))), leaf_input=leaf_input)

            self.tape.append(bwd)
        return y

    # ------------------------------------------------------------------ fused ConvTranspose3d(k2,s2) -> Conv3d
    def _ones(self, like: Act) -> Act:
        """All-ones single-channel activation (the input channel that carries the transposed convolution's bias)."""
        key = (str(self.device), self.tdtype, like.n, like.d, like.h, like.w)
        buf = _ONES.get(key)
        if buf is None:
            buf = torch.zeros((like.n, 1, like.d, like.h, like.w, 8), dtype=self.tdtype, device=self.device)
            buf[..., 0] = 1
            _ONES[key] = buf
        return Act(buf, 1, like.n, like.d, like.h, like.w)

    def up_fusable(self, srcs: Sequence[Act], cout: int, k: int) -> bool:
        """The fused stage needs k in {3, 5} and, in bf16 mode, tcgen05 coverage of the composed convolution
        (forward, weight gradient and every data gradient); fp32 check mode fuses only when forced."""
        if UP_FUSION == "off" or k not in (3, 5) or len(srcs) + 1 > _lib.CTU_MAX_SRC:
            return False
        if UP_FUSION == "force":
            return True
        if self.dtype == CTU_F32 or not self.use_tc:
            return False
        lib = _lib.load()
        chans = [s.c for s in srcs] + [1]
        s0 = srcs[0]
        co8 = lib.ctu_upfuse_cout(cout)
        ca = int_array(chans)
        return bool(lib.ctu_conv_tc_supported(3, len(chans), ca, co8, s0.d, s0.h, s0.w)
                    and lib.ctu_conv_tc_wgrad_supported(3, len(chans), ca, co8, s0.d, s0.h, s0.w)
                    and all(lib.ctu_conv_tc_supported(3, 1, int_array([co8]), s.c, s0.d, s0.h, s0.w) for s in srcs))

    def up_conv(self, srcs: Sequence[Act], ct, cv, k: int, need_src_grad: Sequence[bool], bn_stats: bool) -> Act:
        """conv(convT(cat(srcs))) as one 3x3x3 convolution on the low-resolution grid (csrc/fuse.cu): the 8x larger
        intermediate of models.py:37-38 is never written.  Returns the PHASE-MAJOR output (``c_nat`` set)."""
        lib = _lib.load()
        cin = sum(s.c for s in srcs)
        cout = cv.weight.shape[0]
        co8 = lib.ctu_upfuse_cout(cout)
        has_b3 = cv.bias is not None

        def compose(eng):
            wn = eng.f32(co8, cin + 1, 27)
            b3n = eng.f32(co8) if has_b3 else None
            ws = eng.f32(lib.ctu_upfuse_workspace_floats(cin, cout, k))
            call("ctu_upfuse_compose", ct.weight.data_ptr(), ct.bias.data_ptr() if ct.bias is not None else None,
                 cv.weight.data_ptr(), cv.bias.data_ptr() if has_b3 else None, wn.data_ptr(),
                 b3n.data_ptr() if has_b3 else None, cin, cout, k, ws.data_ptr(), stream_ptr())
            ws.record_stream(torch.cuda.current_stream())
            return wn, b3n

        all_srcs = list(srcs) + [self._ones(srcs[0])]
        self._consume(srcs)
        need = [bool(n) and self.record for n in need_src_grad] + [False]
        wk, tc, wkd, tc_d, wn, extra = self._conv_weights("up_conv", all_srcs, need, None, 3, co8, compose)
        b3n = extra[0]
        y = self._conv_fwd(all_srcs, wk, tc, b3n, 3, co8, cout, bn_stats)
        y.c_nat = cout
        if self.record:
            def bwd():
                dwn = torch.empty_like(wn)
                dbn = self.f32(co8) if has_b3 else None
                dwt, dw3 = self._grad_buffer(ct.weight), self._grad_buffer(cv.weight)
                dbt = self._grad_buffer(ct.bias) if ct.bias is not None else None
                db3 = self._grad_buffer(cv.bias) if has_b3 else None

                def decompose():
                    ws = self.f32(lib.ctu_upfuse_workspace_floats(cin, cout, k))
                    call("ctu_upfuse_decompose", dwn.data_ptr(), dbn.data_ptr() if dbn is not None else None,
                         ct.weight.data_ptr(), ct.bias.data_ptr() if ct.bias is not None else None,
                         cv.weight.data_ptr(), dwt.data_ptr(), dbt.data_ptr() if dbt is not None else None,
                         dw3.data_ptr(), db3.data_ptr() if db3 is not None else None, cin, cout, k, ws.data_ptr(),
                         stream_ptr())
                    for t in (dwn, dbn, ws):
                        if t is not None:
                            t.record_stream(torch.cuda.current_stream())
                    self._pgrad_done(((ct.weight, dwt), (ct.bias, dbt), (cv.weight, dw3), (cv.bias, db3)))

                # a composed 3^3 stage has structurally zero taps (each phase sees 2 of 3 per dimension) that the weight
                # gradient skips; composed from 5^3 every low-resolution tap is populated
                self._conv_bwd(all_srcs, need, wkd, tc_d, y, 3, co8, dwn, dbn, decompose,
                               phase_cout=cout if k == 3 else 0)

            self.tape.append(bwd)
        return y

    def _set_agrad(self, act: Act, g: Act):
        if id(act) in self.agrads:
            raise RuntimeError("internal: activation received two gradients")
        self.agrads[id(act)] = g

    # ------------------------------------------------------------------ ConvTranspose3d k2 s2
    def convt(self, srcs: Sequence[Act], weight, bias, need_src_grad: Sequence[bool]) -> Act:
        cout = weight.shape[1]
        s0 = srcs[0]
        self._consume(srcs)
        pa, ca, ns = self._src_args(srcs)
        lib = _lib.load()
        chans = [s.c for s in srcs]
        need = list(need_src_grad)
        want_bwd = self.record

        def prep(eng):
            # forward weights and (training) the data-gradient weights of every source: parameters only, so they are
            # prepared on the weight-preparation stream with everything else, off the layer chain
            ca_ = int_array(chans)
            wp_ = eng.f32(lib.ctu_convt_wpack_floats(cout, len(chans), ca_))
            call("ctu_convt_pack_weight", weight.data_ptr(), wp_.data_ptr(), cout, len(chans), ca_, stream_ptr())
            out = [wp_]
            for i, c in enumerate(chans):
                if want_bwd and need[i]:
                    wpd_ = eng.f32(lib.ctu_convt_wpack_dgrad_floats(cout, c))
                    call("ctu_convt_pack_weight_dgrad", weight.data_ptr(), wpd_.data_ptr(), cout, len(chans), ca_, i, stream_ptr())
                    out.append(wpd_)
                else:
                    out.append(None)
            return tuple(out)

        res = self._prepared("convt", prep)
        wp, wpds = res[0], list(res[1:])
        y = self.new_act(cout, s0.n, 2 * s0.d, 2 * s0.h, 2 * s0.w)
        call("ctu_convt2_fprop", self.dtype, pa, ca, ns, wp.data_ptr(), bias.data_ptr() if bias is not None else None,
             y.ptr, cout, s0.n, s0.d, s0.h, s0.w, stream_ptr())
        if self.record:
            srcs = list(srcs)

            def bwd():
                dy = self.agrads.pop(id(y))
                pa, ca, ns = self._src_args(srcs)
                if weight.requires_grad:
                    def wgrad():
                        dwp = torch.empty_like(wp)
                        db = self._grad_buffer(bias) if (bias is not None and bias.requires_grad) else None
                        call("ctu_convt2_wgrad", self.dtype, pa, ca, ns, dy.ptr, dwp.data_ptr(),
                             db.data_ptr() if db is not None else None, cout, s0.n, s0.d, s0.h, s0.w, stream_ptr())
                        dw = self._grad_buffer(weight)
                        call("ctu_convt_unpack_wgrad", dwp.data_ptr(), dw.data_ptr(), cout, ns, ca, stream_ptr())
                        self._add_pgrad(weight, dw)
                        if db is not None:
                            self._add_pgrad(bias, db)

                    if WGRAD_ASYNC and CONVT_WGRAD_ASYNC:
                        main = torch.cuda.current_stream()
                        side = _side_stream(self.device, 1)
                        side.wait_stream(main)
                        with torch.cuda.stream(side):
                            wgrad()
                        dy.buf.record_stream(side)
                        for s in srcs:
                            s.buf.record_stream(side)
                        self._wgrad_stream = side
                    else:
                        wgrad()
                for i, s in enumerate(srcs):
                    if not need[i]:
                        continue
                    wpd = wpds[i]
                    dx = self.new_act(s.c, s.n, s.d, s.h, s.w)
                    call("ctu_convt2_dgrad", self.dtype, dy.ptr, wpd.data_ptr(), dx.ptr, cout, s.c,
                         s.n, s.d, s.h, s.w, stream_ptr())
                    self._set_agrad(s, dx)

            self.tape.append(bwd)
        return y

    # ------------------------------------------------------------------ BatchNorm3d + ReLU (+ MaxPool)
    def bn_relu(self, y: Act, bn, training: bool, extra_updates: int = 0, pool: bool = False, keep=None):
        """Returns ``a`` or ``(a, pooled)``.  ``extra_updates``: additional running-stat updates applied
        when the backward pass runs (the reentrant-checkpoint recomputation of the reference).  ``keep``: the float32
        [n, cpad] keep factors of the Dropout3d that follows the ReLU (``dropout_masks``), applied inside the kernels and
        kept for the backward pass: the reference's reentrant checkpoint restores the RNG state, so its recomputation draws
        the same mask and reusing the forward's factors is exact."""
        # nn.BatchNorm3d configurations no preset of the reference uses (models.py:27,31 build BatchNorm3d(c) with the
        # defaults) are refused rather than silently computed differently from torch:
        if bn.momentum is None:
            raise NotImplementedError("BatchNorm3d(momentum=None) (cumulative moving average) is not implemented")
        if bool(bn.training) != bool(training):
            raise NotImplementedError("a BatchNorm3d whose .training flag differs from the network's (frozen BatchNorm "
                                      "inside a training net, or the reverse) is not implemented")
        if not training and (not bn.track_running_stats or bn.running_mean is None or bn.running_var is None):
            raise NotImplementedError("eval-mode BatchNorm3d without running statistics (track_running_stats=False) "
                                      "is not implemented")
        if not bn.affine:
            raise NotImplementedError("BatchNorm3d(affine=False) is not implemented")
        pm = 1 if y.c_nat else 0                     # phase-major input: natural dims are twice the stored ones
        c = y.c_nat if pm else y.c
        cpad = (c + 7) // 8 * 8
        yn, yd, yh, yw = y.n, y.d * (2 if pm else 1), y.h * (2 if pm else 1), y.w * (2 if pm else 1)
        count = float(yn * yd * yh * yw)
        ss = self.f32(4 * cpad)
        sums = None
        st = stream_ptr()
        if training:
            sums = y.sums
            if sums is None:
                sums = self.acc64(2 * cpad)
                call("ctu_bn_stats", self.dtype, y.ptr, c, (8 if pm else 1) | self._pz(sums), y.n, y.spatial, sums.data_ptr(), st)
            track = bn.track_running_stats and bn.running_mean is not None
            mom = float(bn.momentum)
        else:
            call("ctu_bn_finalize", None, count, bn.weight.data_ptr(), bn.bias.data_ptr(), bn.running_mean.data_ptr(),
                 bn.running_var.data_ptr(), None, 0.0, float(bn.eps), c, 0, 0, ss.data_ptr(), st)
        a = self.new_act(c, yn, yd, yh, yw)
        pooled = self.new_act(c, yn, yd // 2, yh // 2, yw // 2) if pool else None
        # Small tensors: finalisation (scale / shift, ss for the backward pass, running statistics) inside the forward kernel,
        # one launch less on the critical path.  Large ones keep the separate 1-block finalize: the per-block prologue
        # (double-precision divide / sqrt + a barrier) costs the short-lived blocks of a 128^3 launch 17 us (ncu: 38 -> 56 us).
        fold = training and yn * yd * yh * yw <= BN_FOLD_MAX_VOXELS
        kp = None
        if keep is not None:
            if pm:
                raise RuntimeError("internal: a phase-major BatchNorm input never precedes a dropout site")
            self._wait_keep()
            kp = keep.data_ptr()
        if training and not fold:
            call("ctu_bn_finalize", sums.data_ptr(), count, bn.weight.data_ptr(), bn.bias.data_ptr(),
                 bn.running_mean.data_ptr() if track else None, bn.running_var.data_ptr() if track else None,
                 bn.num_batches_tracked.data_ptr() if track else None, mom, float(bn.eps), c, 1, 1, ss.data_ptr(), st)
        if fold and kp is not None:
            call("ctu_bn_relu_fwd_train_drop", self.dtype, y.ptr, sums.data_ptr(), count, bn.weight.data_ptr(),
                 bn.bias.data_ptr(), bn.running_mean.data_ptr() if track else None,
                 bn.running_var.data_ptr() if track else None, bn.num_batches_tracked.data_ptr() if track else None, mom,
                 float(bn.eps), 1, ss.data_ptr(), a.ptr, pooled.ptr if pool else None, c, yn, yd, yh, yw, pm, kp, st)
        elif fold:
            call("ctu_bn_relu_fwd_train", self.dtype, y.ptr, sums.data_ptr(), count, bn.weight.data_ptr(), bn.bias.data_ptr(),
                 bn.running_mean.data_ptr() if track else None, bn.running_var.data_ptr() if track else None,
                 bn.num_batches_tracked.data_ptr() if track else None, mom, float(bn.eps), 1, ss.data_ptr(), a.ptr,
                 pooled.ptr if pool else None, c, yn, yd, yh, yw, pm, st)
        elif kp is not None:
            call("ctu_bn_relu_fwd_drop", self.dtype, y.ptr, ss.data_ptr(), a.ptr, pooled.ptr if pool else None,
                 c, yn, yd, yh, yw, pm, kp, st)
        else:
            call("ctu_bn_relu_fwd", self.dtype, y.ptr, ss.data_ptr(), a.ptr, pooled.ptr if pool else None,
                 c, yn, yd, yh, yw, pm, st)
        if self.record:
            if not training:
                raise RuntimeError("backward through eval-mode BatchNorm is not supported by the fused path")
            # (a dropout stage never takes the reduction in the consumer's epilogue: that epilogue knows nothing of keep)
            a.bn = {"y": y, "ss": ss, "pm": pm, "pool": bool(pool), "drop": kp is not None, "consumers": 0, "sums2": None}

            def bwd():
                dA = self.agrads.pop(id(a), None)
                dP = self.agrads.pop(id(pooled), None) if pool else None
                if dA is None and dP is None:
                    raise RuntimeError("internal: BatchNorm stage received no gradient")
                if self._deferred_wgrads and count * ((c + 7) // 8) >= DEFER_WINDOW_VOXELS:
                    self._deferred_wgrads.pop(0)()          # a long HBM-bound window starts: run a held-back weight gradient under it
                st = stream_ptr()
                if extra_updates > 0 and bn.track_running_stats and bn.running_mean is not None:
                    # buffers only (nothing in this step reads them): beside the weight gradients, off the critical path
                    mom = float(bn.momentum)

                    def update():
                        call("ctu_bn_running_update", sums.data_ptr(), count, bn.running_mean.data_ptr(),
                             bn.running_var.data_ptr(), bn.num_batches_tracked.data_ptr(), mom, c, extra_updates,
                             stream_ptr())

                    if WGRAD_ASYNC and LEAF_TAIL_ASYNC:
                        self._leaf_tail(torch.cuda.current_stream(), update, sums)
                    elif WGRAD_ASYNC:
                        side = _side_stream(self.device, 1)
                        side.wait_stream(torch.cuda.current_stream())
                        with torch.cuda.stream(side):
                            update()
                        sums.record_stream(side)
                        self._wgrad_stream = side
                    else:
                        update()
                pA = dA.ptr if dA is not None else None
                pP = dP.ptr if dP is not None else None
                sums2 = a.bn["sums2"]
                a.bn = None                                           # (drop the reference cycle through the closure)
                kq = keep.data_ptr() if keep is not None else None      # (the closure holds the keep factors alive)
                if kq is not None:
                    sums2 = self.acc64(2 * cpad)
                    call("ctu_bn_relu_bwd_reduce_drop", self.dtype, y.ptr, ss.data_ptr(), pA, pP, sums2.data_ptr(),
                         c, yn, yd, yh, yw, pm | self._pz(sums2), kq, st)
                elif sums2 is None or dP is not None:                # not produced by the consumer's epilogue: reduce here
                    sums2 = self.acc64(2 * cpad)
                    call("ctu_bn_relu_bwd_reduce", self.dtype, y.ptr, ss.data_ptr(), pA, pP, sums2.data_ptr(),
                         c, yn, yd, yh, yw, pm | self._pz(sums2), st)
                dy = self.new_act(y.c, y.n, y.d, y.h, y.w)          # same layout as y (phase-major stays phase-major)
                dg, db = self._grad_buffer(bn.weight), self._grad_buffer(bn.bias)
                if kq is not None:
                    call("ctu_bn_relu_bwd_apply_drop", self.dtype, y.ptr, ss.data_ptr(), bn.weight.data_ptr(), pA, pP,
                         sums2.data_ptr(), count, dy.ptr, dg.data_ptr(), db.data_ptr(), c, yn, yd, yh, yw, pm, kq, st)
                else:
                    call("ctu_bn_relu_bwd_apply", self.dtype, y.ptr, ss.data_ptr(), bn.weight.data_ptr(), pA, pP,
                         sums2.data_ptr(), count, dy.ptr, dg.data_ptr(), db.data_ptr(), c, yn, yd, yh, yw, pm, st)
                self._add_pgrad(bn.weight, dg)
                self._add_pgrad(bn.bias, db)
                self._set_agrad(y, dy)

            self.tape.append(bwd)
        return (a, pooled) if pool else a

    # ------------------------------------------------------------------ head
    def head(self, srcs: Sequence[Act], weight, bias, flags: int):
        """last_conv (1x1x1 + bias) + output non-linearities.  Returns fp32 NCDHW tensor(s)."""
        cout = weight.shape[0]
        s0 = srcs[0]
        pa, ca, ns = self._src_args(srcs)
        sp = bool(flags & (_lib.HEAD_SP | _lib.HEAD_SP_SOFTMAX))
        self._consume(srcs)
        if self.label_dst is not None:
            labels, origins, patch, dims = self.label_dst
            if len(labels) != (2 if sp else 1):
                raise ValueError("the %s head produces %d label volume(s)" % ("SP" if sp else "plain", 2 if sp else 1))
            vd, vh, vw = dims if origins is not None else (0, 0, 0)
            call("ctu_head_labels", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags,
                 origins.data_ptr() if origins is not None else None, int(patch), vd, vh, vw, labels[0].data_ptr(),
                 labels[1].data_ptr() if sp else None, s0.n, s0.spatial, stream_ptr())
            return None
        if self.accum_dst is not None:
            acc, origins, patch, dims, wtab = self.accum_dst
            nch = 4 if sp else cout
            if acc.dtype != torch.int64 or acc.numel() != nch * dims[0] * dims[1] * dims[2]:
                raise ValueError("the %s head accumulates into int64 [%d, D, H, W]" % ("SP" if sp else "plain", nch))
            call("ctu_head_accumulate", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags,
                 origins.data_ptr(), int(patch), *dims, wtab.data_ptr(), acc.data_ptr(), s0.n, s0.spatial, stream_ptr())
            return None
        if self.fused_loss is not None:
            return self._head_loss(list(srcs), weight, bias, flags, sp)
        if sp:
            out0 = self.f32(s0.n, 2, s0.d, s0.h, s0.w)
            out1 = self.f32(s0.n, 2, s0.d, s0.h, s0.w)
        else:
            out0, out1 = self.f32(s0.n, cout, s0.d, s0.h, s0.w), None
        call("ctu_head_fwd", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags,
             out0.data_ptr(), out1.data_ptr() if sp else None, s0.n, s0.spatial, stream_ptr())
        if self.record:
            srcs = list(srcs)

            def bwd(g0, g1):
                pa, ca, ns = self._src_args(srcs)
                dsrcs = [self.new_act(s.c, s.n, s.d, s.h, s.w) for s in srcs]
                dw, db = self._grad_buffer(weight), self._grad_buffer(bias)
                p0 = g0.data_ptr() if g0 is not None else None
                p1 = g1.data_ptr() if g1 is not None else None

                # product mode: the SP head's backward pass reads the forward outputs instead of recomputing the
                # sigmoids (fp32 check mode keeps the recomputation: s2 = (s1+s2) - s1 loses a few ulps)
                from_out = HEAD_FROM_OUTPUTS and self.dtype == CTU_BF16
                o0 = out0.data_ptr() if from_out else None
                o1 = out1.data_ptr() if (out1 is not None and from_out) else None

                def params():      # parameter gradients: a leaf, beside the weight gradients (second stream)
                    call("ctu_head_bwd", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags, p0, p1,
                         o0, o1, None, dw.data_ptr(), db.data_ptr(), s0.n, s0.spatial, stream_ptr())
                    self._pgrad_done(((weight, dw), (bias, db)))

                if WGRAD_ASYNC:
                    main = torch.cuda.current_stream()
                    side = _side_stream(self.device, 1)
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        params()
                    for g in (g0, g1):
                        if g is not None:
                            g.record_stream(side)
                    self._wgrad_stream = side
                else:
                    params()
                # source gradients: the critical path
                call("ctu_head_bwd", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags, p0, p1,
                     o0, o1, ptr_array([d.ptr for d in dsrcs]), None, None, s0.n, s0.spatial, stream_ptr())
                for s, d in zip(srcs, dsrcs):
                    self._set_agrad(s, d)

            self.head_bwd = bwd
        return (out0, out1) if sp else out0

    def _head_loss(self, srcs, weight, bias, flags, sp):
        """Head + Dice / CrossEntropy in one pass over the sources (training step only): see csrc/head.cu."""
        targets, softmax_for_dice, ce_l, dice_l, comps, mirror = self.fused_loss
        cout = weight.shape[0]
        s0 = srcs[0]
        targets = list(targets) if isinstance(targets, (tuple, list)) else [targets]
        if len(targets) != (2 if sp else 1):
            raise ValueError("the %s head takes %d target tensor(s), got %d" % ("SP" if sp else "plain", 2 if sp else 1, len(targets)))
        want = (s0.n, 2 if sp else cout, s0.d, s0.h, s0.w)
        u8 = int(targets[0].dtype == torch.uint8)
        if u8:                              # label masks [B, D, H, W] (two classes), 1 byte per voxel instead of 8
            want = (s0.n, s0.d, s0.h, s0.w)
            if not sp and cout != 2:
                raise TypeError("uint8 mask targets need a two-class output")
        for t in targets:
            if (tuple(t.shape) != want or t.dtype != (torch.uint8 if u8 else torch.float32) or not t.is_contiguous()
                    or t.device != s0.buf.device):
                raise TypeError("targets: contiguous float32 one-hot tensors [B, C, D, H, W] or uint8 label masks [B, D, H, W] "
                                "on %s (expected shape %s)" % (s0.buf.device, want))
            if t.data_ptr() % (2 if u8 else 8):
                # the kernels read two voxels per load (csrc/head.cu, head_load_targets2)
                raise TypeError("targets: a %s target must start %d-byte aligned (a contiguous view at offset %d elements "
                                "is not)" % (t.dtype, 2 if u8 else 8, t.storage_offset()))
        pa, ca, ns = self._src_args(srcs)
        t0, t1 = targets[0].data_ptr(), (targets[1].data_ptr() if sp else None)
        sums = self.f64(4 * len(targets) * s0.n)
        call("ctu_head_loss_fwd", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags, t0, t1, u8,
             int(softmax_for_dice), float(ce_l), float(dice_l), sums.data_ptr(), comps.data_ptr(),
             mirror.data_ptr() if mirror is not None else None, s0.n, s0.spatial, stream_ptr())
        if self.record:
            def bwd(g0=None, g1=None):
                pa, ca, ns = self._src_args(srcs)
                dsrcs = [self.new_act(s.c, s.n, s.d, s.h, s.w) for s in srcs]
                dw, db = self._grad_buffer(weight), self._grad_buffer(bias)
                dlc = self.f32(s0.n, cout, s0.d, s0.h, s0.w)
                # source gradients (the critical path); the logit gradients are kept for the parameter gradients
                call("ctu_head_loss_bwd", self.dtype, pa, ca, ns, weight.data_ptr(), bias.data_ptr(), cout, flags, t0, t1, u8,
                     int(softmax_for_dice), float(ce_l), float(dice_l), sums.data_ptr(), ptr_array([d.ptr for d in dsrcs]),
                     dlc.data_ptr(), s0.n, s0.spatial, stream_ptr())
                for s, d in zip(srcs, dsrcs):
                    self._set_agrad(s, d)

                def params():      # parameter gradients: a leaf, beside the weight gradients (second stream)
                    call("ctu_head_param_grad", self.dtype, pa, ca, ns, dlc.data_ptr(), cout, dw.data_ptr(), db.data_ptr(),
                         s0.n, s0.spatial, stream_ptr())
                    self._pgrad_done(((weight, dw), (bias, db)))

                if WGRAD_ASYNC and LEAF_TAIL_ASYNC and HEAD_PGRAD_LATE:
                    # enqueued when the whole chain has been: it then runs beside the LAST weight gradients (tcgen05 kernels with
                    # a small register footprint) instead of taking the SMs from the BatchNorm kernels at the head of the chain
                    self._late_leaves.append((params, dlc))
                elif WGRAD_ASYNC and LEAF_TAIL_ASYNC:
                    self._leaf_tail(torch.cuda.current_stream(), params, dlc)       # a CUDA-core kernel: not on the tcgen05 stream
                elif WGRAD_ASYNC:
                    main = torch.cuda.current_stream()
                    side = _side_stream(self.device, 1)
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        params()
                    dlc.record_stream(side)
                    self._wgrad_stream = side
                else:
                    params()

            self.head_bwd = bwd
        return None

    # ------------------------------------------------------------------ backward driver
    def run_tape(self):
        """Run the recorded backward closures (last stage first) and join the weight-gradient stream."""
        for fn in reversed(self.tape):
            fn()
        self.tape = []
        for fn, keep in self._late_leaves:
            self._leaf_tail(torch.cuda.current_stream(), fn, keep)
        self._late_leaves = []
        while self._deferred_wgrads:
            self._deferred_wgrads.pop(0)()
        if self._wgrad_stream is not None:                   # weight gradients -> visible to the optimizer's stream
            torch.cuda.current_stream().wait_stream(self._wgrad_stream)
            self._wgrad_stream = None
        if self._input_grad_stream is not None:
            torch.cuda.current_stream().wait_stream(self._input_grad_stream)
            self._input_grad_stream = None
        if self._leaf_tail_stream is not None:
            torch.cuda.current_stream().wait_stream(self._leaf_tail_stream)
            self._leaf_tail_stream = None

    def backward(self, g0=None, g1=None):
        # (drop the closure first: it references the engine AND the forward outputs, i.e. the autograd graph -- a cycle
        # that would keep this pass's AccumulateGrad nodes alive until the next garbage collection)
        fn, self.head_bwd = self.head_bwd, None
        fn(g0, g1)
        self.run_tape()


# The weight-streaming kernel (conv_wide.cu) is preferred over the resident-weights kernel where both cover a layer
# and the grid is small (h and w at most WIDE_MAX_HW): measured on B200 (scripts/bench_wide.py, batch 4) 56->56 3^3 at
# 16^3 takes 10.9 us streamed vs 32.0 us resident, while at 32^3 the resident kernel wins (28->28: 24.8 vs 29.3 us).
WIDE_MIN_CH = 9
WIDE_MAX_HW = 16


def tc_variant(k, src_channels, cout, n, d, h, w) -> int:
    """Which tcgen05 kernel runs conv(cat(srcs)) -> cout: 0 none (CUDA cores), 1 conv_tc.cu, 2 conv_wide.cu."""
    lib = _lib.load()
    chans = list(src_channels)
    narrow = bool(lib.ctu_conv_tc_supported(k, len(chans), int_array(chans), cout, d, h, w))
    if len(chans) == 1 and lib.ctu_conv_wide_supported(k, chans[0], cout, n, d, h, w):
        if not narrow or (min(chans[0], cout) >= WIDE_MIN_CH and max(h, w) <= WIDE_MAX_HW):
            return 2
    return 1 if narrow else 0


def wgrad_variant(k, src_channels, cout, d, h, w, phase_cout=0) -> int:
    """Which kernel computes the weight gradient of conv(cat(srcs)) -> cout on the tensor path: 0 none (CUDA cores),
    1 conv_tc.cu (16-wide rows), 2 the tap-stationary small-grid kernel (8 x 8 plane tiles, d-planes split over CTAs)."""
    lib = _lib.load()
    chans = list(src_channels)
    small = len(chans) == 1 and not phase_cout and lib.ctu_conv_wide_wgrad_supported(k, chans[0], cout, d, h, w)
    if small and max(h, w) <= WIDE_MAX_HW:
        return 2
    if lib.ctu_conv_tc_wgrad_supported(k, len(chans), int_array(chans), cout, d, h, w):
        return 1
    return 2 if small else 0


def tc_supported(k, src_channels, cout, d, h, w) -> bool:
    """Shapes covered by the tcgen05 implicit-GEMM convolution (the predicate lives in conv_tc.cu)."""
    if not 1 <= len(src_channels) <= _lib.CTU_MAX_SRC:
        return False
    return bool(_lib.load().ctu_conv_tc_supported(k, len(src_channels), int_array(list(src_channels)), cout, d, h, w))
