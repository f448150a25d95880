"""GPU CT preprocessing and sliding-window inference (BASELINE.json configs 4 and 5).

The reference has NO implementation of HU windowing, thresholding, resampling or patch-wise
inference (SURVEY.md section 8c: they live in the author's separate ``headctools`` project); the
semantics implemented here are the ones frozen in ``oracle/unet_oracle.py`` (clamp + rescale,
``>=`` threshold, PyTorch 'nearest' / 'trilinear, align_corners=False' resampling, non-overlapping
patch grid) -- parity with the reference is therefore unpinned by construction.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from ._lib import call, load, stream_ptr
from .utilities import hard_segm_from_tensor


def _vol(t, dtype, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s runs on CUDA tensors only (no CPU fallback)" % what)
    if t.dim() != 3:
        raise ValueError("%s expects a [D, H, W] volume" % what)
    if t.dtype != dtype:
        raise TypeError("%s expects %s, got %s" % (what, dtype, t.dtype))
    return t.contiguous()


def hu_window(hu: torch.Tensor, lo: float, hi: float) -> torch.Tensor:
    """int16 HU -> float32 in [0, 1]: (clamp(hu, lo, hi) - lo) / (hi - lo)."""
    hu = _vol(hu, torch.int16, "hu_window")
    out = torch.empty(hu.shape, dtype=torch.float32, device=hu.device)
    call("ctu_hu_window", hu.data_ptr(), out.data_ptr(), hu.numel(), float(lo), float(hi), stream_ptr())
    return out


def hu_threshold(hu: torch.Tensor, thr: int) -> torch.Tensor:
    """int16 HU -> uint8 bone mask (hu >= thr)."""
    hu = _vol(hu, torch.int16, "hu_threshold")
    out = torch.empty(hu.shape, dtype=torch.uint8, device=hu.device)
    call("ctu_hu_threshold", hu.data_ptr(), out.data_ptr(), hu.numel(), int(thr), stream_ptr())
    return out


# ------------------------------------------------------------------------------------------------ connected components
# Semantics (DESIGN.md section 7c; frozen by tests/components_oracle.py on top of scipy.ndimage.label): a voxel is
# foreground when it is non-zero; connectivity 6 / 18 / 26 = generate_binary_structure(3, 1 / 2 / 3); components are
# numbered 1..n per volume in the raster order of their first voxel (scipy's numbering).  Each volume of a [B, D, H, W]
# input is labelled on its own.  No host synchronisation: counts stay on the device.
_MASK_DTYPES = {torch.uint8: 1, torch.bool: 1, torch.float32: 4}      # CTU_MASK_U8 / CTU_MASK_F32
_CONNECTIVITIES = (6, 18, 26)


def _components_input(mask, connectivity, what):
    """[B, D, H, W] contiguous view of ``mask`` and the C-ABI dtype code; every argument error raises before a launch."""
    if connectivity not in _CONNECTIVITIES:
        raise ValueError("%s: connectivity must be 6, 18 or 26, got %r" % (what, connectivity))
    if not isinstance(mask, torch.Tensor):
        raise RuntimeError("%s runs on CUDA tensors only (no CPU fallback)" % what)
    if mask.dim() not in (3, 4):
        raise ValueError("%s expects a [D, H, W] or [B, D, H, W] volume, got %d dimensions" % (what, mask.dim()))
    if mask.dtype not in _MASK_DTYPES:
        raise TypeError("%s expects uint8, bool or float32, got %s" % (what, mask.dtype))
    if mask.numel() >= 2 ** 31:
        raise ValueError("%s: %d voxels; B*D*H*W must be below 2^31" % (what, mask.numel()))
    if not mask.is_cuda:
        raise RuntimeError("%s runs on CUDA tensors only (no CPU fallback)" % what)
    m = mask.contiguous()
    return (m if m.dim() == 4 else m.unsqueeze(0)), _MASK_DTYPES[mask.dtype]


def _components_workspace(m):
    nbytes = load().ctu_components_workspace_bytes(*m.shape)
    return torch.empty(nbytes, dtype=torch.uint8, device=m.device), nbytes


def label_components(mask: torch.Tensor, connectivity: int = 6):
    """``scipy.ndimage.label`` on the device: (labels int32 like ``mask``, counts int64 [B] -- 0-dim for a [D, H, W]
    input -- the number of components per volume).  ``mask``: uint8, bool or float32 CUDA tensor."""
    m, code = _components_input(mask, connectivity, "label_components")
    labels = torch.empty(m.shape, dtype=torch.int32, device=m.device)
    counts = torch.zeros(m.shape[0], dtype=torch.int64, device=m.device)
    if m.numel():
        ws, nbytes = _components_workspace(m)
        call("ctu_label_components", code, m.data_ptr(), *m.shape, connectivity, labels.data_ptr(), counts.data_ptr(),
             ws.data_ptr(), nbytes, stream_ptr())
    if mask.dim() == 3:
        return labels[0], counts[0]
    return labels, counts


def _filter_components(mask, connectivity, min_size, what):
    m, code = _components_input(mask, connectivity, what)
    out = torch.empty_like(m)
    if m.numel():
        ws, nbytes = _components_workspace(m)
        call("ctu_filter_components", code, m.data_ptr(), *m.shape, connectivity, min_size, out.data_ptr(), ws.data_ptr(),
             nbytes, stream_ptr())
    return out.view(mask.shape)


def largest_component(mask: torch.Tensor, connectivity: int = 6) -> torch.Tensor:
    """``mask`` with every voxel outside the largest component of its volume set to 0 (ties: the component whose first
    voxel comes first in raster order, i.e. the lower label).  Same dtype and shape; an empty volume stays empty."""
    return _filter_components(mask, connectivity, -1, "largest_component")


def remove_small_components(mask: torch.Tensor, min_size: int, connectivity: int = 6) -> torch.Tensor:
    """``mask`` with the voxels of every component smaller than ``min_size`` voxels set to 0.  Same dtype and shape."""
    if int(min_size) != min_size or min_size < 0:
        raise ValueError("remove_small_components: min_size must be a non-negative integer, got %r" % (min_size,))
    return _filter_components(mask, connectivity, int(min_size), "remove_small_components")


def resample_nearest(vol: torch.Tensor, out_size) -> torch.Tensor:
    """PyTorch 'nearest' semantics: src = min(floor(dst * in/out), in - 1) per axis (float32 scale)."""
    if vol.dtype not in (torch.float32, torch.uint8):
        raise TypeError("resample_nearest expects float32 or uint8")
    vol = _vol(vol, vol.dtype, "resample_nearest")
    out = torch.empty(tuple(out_size), dtype=vol.dtype, device=vol.device)
    fn = "ctu_resample_nearest_f32" if vol.dtype == torch.float32 else "ctu_resample_nearest_u8"
    call(fn, vol.data_ptr(), out.data_ptr(), *vol.shape, *out.shape, stream_ptr())
    return out


def nearest_source_index(out_size: int, in_size: int, device="cuda") -> torch.Tensor:
    idx = torch.empty(out_size, dtype=torch.int32, device=device)
    call("ctu_resample_nearest_index", idx.data_ptr(), out_size, in_size, stream_ptr())
    return idx


def resample_trilinear(vol: torch.Tensor, out_size) -> torch.Tensor:
    """F.interpolate(mode='trilinear', align_corners=False) semantics, float32."""
    vol = _vol(vol, torch.float32, "resample_trilinear")
    out = torch.empty(tuple(out_size), dtype=torch.float32, device=vol.device)
    call("ctu_resample_trilinear_f32", vol.data_ptr(), out.data_ptr(), *vol.shape, *out.shape, stream_ptr())
    return out


def _captured_patch_labels(model, xb: torch.Tensor):
    """Eval-mode forward + argmax of one patch batch, replayed from a CUDA graph captured per (model, batch shape): an
    inference pass is ~110 launches with no host synchronisation, and at small patch batches the Python / ctypes dispatch
    (about 2 ms) is longer than the GPU work."""
    graphs = model.__dict__.setdefault("_infer_graphs", {})       # lives and dies with the model
    key = (tuple(xb.shape), str(xb.device), getattr(model, "compute_dtype", None))
    ent = graphs.get(key)
    weights = list(model.parameters()) + list(model.buffers())
    if ent is not None and (len(ent[3]) != len(weights) or any(a is not b for a, b in zip(ent[3], weights))):
        ent = None            # a parameter / buffer OBJECT was replaced: the capture reads the old storage
    if ent is None:
        static_in = torch.empty_like(xb)
        static_in.copy_(xb)

        def run():
            o = model(static_in)
            o = o if isinstance(o, tuple) else (o,)
            return [hard_segm_from_tensor(ok) for ok in o]

        run()                                   # warm-up: weight-preparation plan, allocator pools
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            outs = run()
        ent = (g, static_in, outs, weights)
        graphs[key] = ent
        if len(graphs) > 8:                     # a handful of shapes at most: drop the oldest capture
            graphs.pop(next(iter(graphs)))
    g, static_in, outs, _ = ent
    static_in.copy_(xb)
    g.replay()
    return outs


def _captured_fused_pass(model, vol, patch, batch, n_out, accum=None):
    """(static volume, static outputs, static origins [batch, 3], graph) of one fused patch-batch pass, captured once per
    (model weights, volume shape, patch, batch, pass kind).  ``accum`` None: gather -> network -> labels scattered at the
    origins; the static outputs are the label volumes.  ``accum`` = (blend, sigma_scale, channels): gather -> network ->
    weighted head outputs added to the accumulators (``model.accumulate_windows``); the static outputs are
    [int64 accumulators [channels, D, H, W], float32 weight table [3, patch]]."""
    graphs = model.__dict__.setdefault("_infer_graphs", {})
    kind = "fused" if accum is None else ("accumulate", accum[0], float(accum[1]))
    key = (kind, tuple(vol.shape), str(vol.device), int(patch), int(batch), getattr(model, "compute_dtype", None))
    weights = list(model.parameters()) + list(model.buffers())
    ent = graphs.get(key)
    if ent is not None and (len(ent[4]) != len(weights) or any(a is not b for a, b in zip(ent[4], weights))):
        ent = None
    if ent is None:
        st_vol = vol.clone()
        st_org = torch.zeros((batch, 3), dtype=torch.int32, device=vol.device)
        if accum is None:
            st_outs = [torch.zeros(tuple(vol.shape[1:]), dtype=torch.float32, device=vol.device) for _ in range(n_out)]

            def run():
                model.predict_labels(vol=st_vol, origins=st_org, patch=patch, out=st_outs)
        else:
            wt = torch.tensor(window_weights(patch, accum[0], accum[1]), dtype=torch.float32)
            st_outs = [torch.zeros((accum[2],) + tuple(vol.shape[1:]), dtype=torch.int64, device=vol.device),
                       wt.expand(3, patch).contiguous().to(vol.device)]

            def run():
                model.accumulate_windows(vol=st_vol, origins=st_org, patch=patch, weights=st_outs[1], acc=st_outs[0])
        run()                                   # warm-up: plans, allocator pools
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            run()
        ent = (st_vol, st_outs, st_org, g, weights)
        graphs[key] = ent
        if len(graphs) > 8:
            graphs.pop(next(iter(graphs)))
    return ent[:4]


@torch.no_grad()
def sliding_window_argmax(model, vol: torch.Tensor, patch: int = 128, batch: int = 4, graph: bool = True, fused: bool = True,
                          rank: int = 0, world: int = 1, group=None):
    """Eval-mode model over the non-overlapping ``patch``^3 grid of ``vol`` [Cin, D, H, W]; returns the
    stitched float32 label volume(s) (one per model output), as ``hard_segm_from_tensor`` would label
    each patch (utilities.py:103-124).

    ``fused`` (the B200 modules): per patch batch ONE gather kernel builds the blocked input from ``vol`` at the patch
    origins and the head kernel writes the hard labels straight into the full-size output volumes
    (``model.predict_labels``) -- no slicing / stacking, no fp32 [B,2,p,p,p] outputs, no separate argmax, no stitch copies.
    Otherwise: slices stacked on the host side of the API and (``graph``) every full patch batch replayed from a captured
    CUDA graph.  ``world`` > 1: the patches are sharded over the ranks (``parallel.shard_range``, no data-path collective in
    the forward passes) and the disjoint label patches are merged by one all-reduce of the label volumes."""
    if vol.dim() != 4:
        raise ValueError("expected [Cin, D, H, W]")
    c, d, h, w = vol.shape
    if d % patch or h % patch or w % patch:
        raise ValueError("volume %s must be a multiple of the patch size %d" % ((d, h, w), patch))
    was_training = model.training
    model.eval()
    origins = [(z, y, x) for z in range(0, d, patch) for y in range(0, h, patch) for x in range(0, w, patch)]
    if world > 1:
        from .parallel import shard_range
        lo, hi = shard_range(len(origins), rank, world)
        origins = origins[lo:hi]
    outs = None
    if fused and vol.is_cuda and hasattr(model, "predict_labels") and vol.dtype == torch.float32:
        vol = vol.contiguous()
        n_out = 2 if getattr(model, "_head_mode", "plain") != "plain" else 1
        org = torch.tensor(origins, dtype=torch.int32, device=vol.device).view(-1, 3)
        nfull = (len(origins) // batch) * batch if graph else 0
        if nfull:
            # one captured graph per (volume shape, patch, batch): ~110 launches per patch batch are host-bound below batch 8
            st_vol, st_outs, st_org, g = _captured_fused_pass(model, vol, patch, batch, n_out)
            if st_vol.data_ptr() != vol.data_ptr():
                st_vol.copy_(vol)
            if world > 1:
                for o in st_outs:
                    o.zero_()
            for i in range(0, nfull, batch):
                st_org.copy_(org[i:i + batch])
                g.replay()
            for i in range(nfull, len(origins), batch):          # a ragged last batch runs eagerly on the same buffers
                model.predict_labels(vol=st_vol, origins=org[i:i + batch], patch=patch, out=st_outs)
            outs = [o.clone() for o in st_outs]                   # the static buffers belong to the capture
        else:
            alloc = torch.zeros if world > 1 else torch.empty
            outs = [alloc((d, h, w), dtype=torch.float32, device=vol.device) for _ in range(n_out)]
            for i in range(0, len(origins), batch):
                model.predict_labels(vol=vol, origins=org[i:i + batch], patch=patch, out=outs)
    else:
        for i in range(0, len(origins), batch):
            chunk = origins[i:i + batch]
            xb = torch.stack([vol[:, z:z + patch, y:y + patch, x:x + patch] for z, y, x in chunk]).contiguous()
            if graph and vol.is_cuda:
                labs = _captured_patch_labels(model, xb)
            else:
                o = model(xb)
                o = o if isinstance(o, tuple) else (o,)
                labs = [hard_segm_from_tensor(ok) for ok in o]
            if outs is None:
                alloc = torch.zeros if world > 1 else torch.empty
                outs = [alloc((d, h, w), dtype=torch.float32, device=vol.device) for _ in labs]
            for k, lab in enumerate(labs):
                for j, (z, y, x) in enumerate(chunk):
                    outs[k][z:z + patch, y:y + patch, x:x + patch] = lab[j]
    if world > 1:
        import torch.distributed as dist
        if outs is None:                      # a rank without patches still takes part in the merge
            n_out = 2 if getattr(model, "_head_mode", "plain") != "plain" else 1
            outs = [torch.zeros((d, h, w), dtype=torch.float32, device=vol.device) for _ in range(n_out)]
        for o in outs:
            dist.all_reduce(o, op=dist.ReduceOp.SUM, group=group)     # disjoint supports: the sum IS the stitch
    model.train(was_training)
    return outs


# ------------------------------------------------------------------------------------------------ overlapping windows
# Semantics (DESIGN.md section 7b; frozen by tests/window_oracle.py -- the reference has no sliding-window code):
#   grid     per axis of size S, patch p, overlap in [0, 1): step = max(1, floor(p (1 - overlap))); one origin 0 when S <= p
#            (the window reaches past the volume: its inputs there read as 0, its outputs there are dropped), otherwise
#            ceil((S - p) / step) + 1 origins min(i step, S - p); the windows are the z-major product of the axis lists.
#   weights  separable w(z, y, x) = wz[z] wy[y] wx[x]; "constant": 1; "gaussian": max(g(t) / max g, 2^-6) with
#            g(t) = exp(-(t - (p - 1) / 2)^2 / (2 sigma^2)), sigma = sigma_scale p.
#   sums     every window voxel inside the volume adds llrint(w v 2^40) to an int64 accumulator per head output channel
#            value v (in [0, 2]): exact integer sums, independent of batch, window order and ranks.
#   outputs  labels = argmax over the accumulators (first maximum wins); probabilities = acc 2^-40 / (Nz[z] Ny[y] Nx[x]),
#            Na[t] = sum of wa[t - o] over the axis origins o whose window covers t.
ACC_FRACTION_BITS = 40
_BLENDS = ("constant", "gaussian")


def window_origins(size: int, patch: int, overlap: float):
    """Window origins along one axis of ``size`` voxels (see the grid rule above)."""
    step = max(1, int(math.floor(patch * (1.0 - overlap))))
    if size <= patch:
        return [0]
    n = -(-(size - patch) // step) + 1
    return [min(i * step, size - patch) for i in range(n)]


def window_weights(patch: int, blend: str = "gaussian", sigma_scale: float = 0.125):
    """float64 [patch] weight table of one axis.  The 2^-6 floor keeps the 3-D weight >= 2^-18, so a voxel's total
    weight stays far above the 2^-40 fixed-point resolution of the accumulators."""
    if blend == "constant":
        return np.ones(patch, dtype=np.float64)
    if blend != "gaussian":
        raise ValueError("blend must be one of %s, got %r" % (_BLENDS, blend))
    sigma = sigma_scale * patch
    t = np.arange(patch, dtype=np.float64)
    g = np.exp(-((t - (patch - 1) / 2.0) ** 2) / (2.0 * sigma * sigma))
    return np.maximum(g / g.max(), 2.0 ** -6)


def window_normaliser(size: int, patch: int, origins, weights):
    """float64 [size] total weight Na[t] of one axis: the sum of weights[t - o] over the origins o whose window covers t."""
    n = np.zeros(size, dtype=np.float64)
    for o in origins:
        hi = min(o + patch, size)
        n[o:hi] += np.asarray(weights, dtype=np.float64)[:hi - o]
    return n


def window_grid(shape, patch: int, overlap: float):
    """Per-axis origin lists of a [D, H, W] volume.  Raises OverflowError when the most-covered voxel could overflow the
    int64 accumulators: each window adds at most 2 * 2^40 (weight <= 1, head output <= 2)."""
    axes = [window_origins(int(s), patch, overlap) for s in shape]
    coverage = 1
    for s, org in zip(shape, axes):
        cover = np.zeros(int(s), dtype=np.int64)
        for o in org:
            cover[o:o + patch] += 1
        coverage *= int(cover.max())
    if coverage * 2 ** (ACC_FRACTION_BITS + 1) >= 2 ** 63:
        raise OverflowError("a voxel is covered by %d windows (patch %d, overlap %g): the fixed-point sums could overflow "
                            "int64; use a smaller overlap" % (coverage, patch, overlap))
    return axes


def _first_conv_in(model):
    return next(m.in_channels for m in model.modules() if isinstance(m, torch.nn.Conv3d))


def _accumulate_windows(model, vol, patch, overlap, blend, sigma_scale, batch, graph, rank, world):
    """Blended int64 accumulators [n_out * channels, D, H, W] of this rank's share of the windows (before any merge),
    and the per-axis origin lists.  With ``graph`` the result is the static buffer of the captured pass: valid until the
    next pass with the same configuration."""
    d, h, w = vol.shape[1:]
    axes = window_grid((d, h, w), patch, overlap)
    origins = [(z, y, x) for z in axes[0] for y in axes[1] for x in axes[2]]
    if world > 1:
        from .parallel import shard_range
        lo, hi = shard_range(len(origins), rank, world)
        origins = origins[lo:hi]
    sp = getattr(model, "_head_mode", "plain") != "plain"
    nch = 4 if sp else model.last_conv.out_channels          # [out][channel]: SP heads have two outputs of two channels
    org = torch.tensor(origins, dtype=torch.int32, device=vol.device).view(-1, 3)
    nfull = (len(origins) // batch) * batch if graph else 0
    if nfull:
        st_vol, (acc, wt), st_org, g = _captured_fused_pass(model, vol, patch, batch, 2 if sp else 1,
                                                            accum=(blend, sigma_scale, nch))
        if st_vol.data_ptr() != vol.data_ptr():
            st_vol.copy_(vol)
    else:
        st_vol, g = vol, None
        acc = torch.empty((nch, d, h, w), dtype=torch.int64, device=vol.device)
        wt = torch.tensor(window_weights(patch, blend, sigma_scale), dtype=torch.float32).expand(3, patch).contiguous()
        wt = wt.to(vol.device)
    acc.zero_()
    for i in range(0, nfull, batch):
        st_org.copy_(org[i:i + batch])
        g.replay()
    for i in range(nfull, len(origins), batch):          # a ragged last batch (or every batch without graph) runs eagerly
        model.accumulate_windows(vol=st_vol, origins=org[i:i + batch], patch=patch, weights=wt, acc=acc)
    return acc, axes


@torch.no_grad()
def sliding_window_predict(model, vol: torch.Tensor, patch: int = 128, overlap: float = 0.5, blend: str = "gaussian",
                           sigma_scale: float = 0.125, batch: int = 4, graph: bool = True, probs: bool = False,
                           rank: int = 0, world: int = 1, group=None):
    """Eval-mode model over overlapping ``patch``^3 windows of ``vol`` float32 CUDA [Cin, D, H, W] of any size, the head
    outputs blended with a constant or Gaussian importance map (semantics above).  Returns the float32 [D, H, W] label
    volume(s), one per model output, as ``sliding_window_argmax`` does; with ``probs`` also returns the normalised blended
    outputs, float32 [C, D, H, W] per output: ``(labels, probs)``.

    Every full batch of windows replays one captured pass (gather -> network -> weighted sums into int64 accumulators),
    a ragged tail runs eagerly, and one kernel finalizes.  ``world`` > 1: the windows are sharded over the ranks
    (``parallel.shard_range``) and one all-reduce of the integer accumulators merges them, so every rank returns exactly
    the single-rank result."""
    if not isinstance(vol, torch.Tensor) or not vol.is_cuda:
        raise RuntimeError("sliding_window_predict runs on CUDA tensors only (no CPU fallback)")
    if vol.dtype != torch.float32:
        raise TypeError("sliding_window_predict expects a float32 volume, got %s" % vol.dtype)
    if vol.dim() != 4:
        raise ValueError("expected [Cin, D, H, W]")
    if not hasattr(model, "accumulate_windows"):
        raise TypeError("sliding_window_predict needs a ctunet_b200 model (got %s)" % type(model).__name__)
    if not 0.0 <= overlap < 1.0:
        raise ValueError("overlap must be in [0, 1), got %r" % (overlap,))
    if blend not in _BLENDS:
        raise ValueError("blend must be one of %s, got %r" % (_BLENDS, blend))
    if not sigma_scale > 0:
        raise ValueError("sigma_scale must be > 0, got %r" % (sigma_scale,))
    m = max(2 ** model._levels(), 4)
    if patch <= 0 or patch % m:
        raise ValueError("patch size %d must be a positive multiple of %d" % (patch, m))
    if batch < 1:
        raise ValueError("batch must be >= 1")
    if vol.shape[0] != _first_conv_in(model):
        raise ValueError("the volume has %d channels, the model takes %d" % (vol.shape[0], _first_conv_in(model)))
    was_training = model.training
    model.eval()
    try:
        vol = vol.contiguous()
        acc, axes = _accumulate_windows(model, vol, patch, overlap, blend, sigma_scale, batch, graph, rank, world)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)     # integer sums: the merge is exact
        d, h, w = vol.shape[1:]
        n_out = 2 if getattr(model, "_head_mode", "plain") != "plain" else 1
        nch = acc.shape[0] // n_out
        labels = [torch.empty((d, h, w), dtype=torch.float32, device=vol.device) for _ in range(n_out)]
        blended, norm = [], None
        if probs:
            wt = window_weights(patch, blend, sigma_scale).astype(np.float32).astype(np.float64)   # the kernel's weights
            norm = torch.from_numpy(np.concatenate([window_normaliser(s, patch, o, wt) for s, o in zip((d, h, w), axes)]))
            norm = norm.to(vol.device)
            blended = [torch.empty((nch, d, h, w), dtype=torch.float32, device=vol.device) for _ in range(n_out)]
        call("ctu_window_finalize", acc.data_ptr(), n_out, nch, d, h, w, norm.data_ptr() if probs else None,
             labels[0].data_ptr(), labels[1].data_ptr() if n_out == 2 else None,
             blended[0].data_ptr() if probs else None, blended[1].data_ptr() if probs and n_out == 2 else None, stream_ptr())
    finally:
        model.train(was_training)
    return (labels, blended) if probs else labels
