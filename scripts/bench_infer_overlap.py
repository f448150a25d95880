"""Overlapping sliding-window inference (preprocess.sliding_window_predict, DESIGN.md section 7b) on one GPU.

  volumes   the 256 x 512 x 512 phantom of scripts/bench_infer.py (bone mask + atlas, 2 channels) and its first 224 slices
            (224 x 512 x 512, a shape sliding_window_argmax refuses at the 128^3 patch)
  sweep     overlap 0 / 0.25 / 0.5, constant / Gaussian blending, patch batch 4 / 8, eval-mode UNetSP (bf16): ms per
            volume, windows, Gvox/s of input voxels
  kernels   one eager pass per volume under torch.profiler (a run of its own): head_accum_kernel, window_finalize_kernel,
            the accumulator zeroing and the patch gather, with achieved GB/s against 6552 GB/s (the copy bandwidth
            measured on this machine type, DESIGN.md)
  baseline  overlap 0 / constant against sliding_window_argmax on the aligned 256 x 512 x 512 volume, same batch

    python scripts/bench_infer_overlap.py [--out FILE]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import ctunet_b200 as C
from ctunet_b200 import preprocess as P

HBM_GBS = 6552.0
PATCH = 128

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None, help="also write the report to this file")
args = ap.parse_args()
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


dev = torch.device("cuda:0")
torch.cuda.set_device(dev)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True)
say("GPU: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(dev), q.stdout.strip() or "unavailable"))


def timeit(fn, reps=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps * 1e-3


# the phantom of scripts/bench_infer.py, thresholded to the bone mask, plus a random atlas channel
D, H, W = 256, 512, 512
g = torch.Generator(device=dev).manual_seed(0)
lin = [torch.linspace(-1, 1, n, device=dev) for n in (D, H, W)]
zz, yy, xx = torch.meshgrid(*lin, indexing="ij")
r = torch.sqrt((zz / 0.8) ** 2 + (yy / 0.88) ** 2 + (xx / 0.72) ** 2)
hu = torch.full((D, H, W), -1000, dtype=torch.int16, device=dev)
hu[r <= 1.0] = 40
hu[(r >= 0.93) & (r <= 1.0)] = 1000
hu = (hu.float() + 30 * torch.randn(hu.shape, device=dev, generator=g)).clamp(-1024, 3071).to(torch.int16)
del zz, yy, xx, r
bone = P.hu_threshold(hu, 300)
atlas = (torch.rand(D, H, W, device=dev, generator=g) > 0.8).float()
vol256 = torch.stack((bone.float(), atlas)).contiguous()
vol224 = vol256[:, :224].contiguous()
del hu, bone, atlas

torch.manual_seed(0)
net = C.UNetSP().to(dev).eval()


def windows(shape, overlap):
    n = 1
    for s in shape:
        n *= len(P.window_origins(s, PATCH, overlap))
    return n


say("\n== sliding_window_predict, UNetSP bf16, patch %d (labels only; CUDA events, 3 timed passes after 1 warm-up)" % PATCH)
for name, vol in (("256x512x512", vol256), ("224x512x512", vol224)):
    vox = vol[0].numel()
    for overlap in (0.0, 0.25, 0.5):
        for blend in ("constant", "gaussian"):
            for batch in (4, 8):
                t = timeit(lambda: P.sliding_window_predict(net, vol, patch=PATCH, overlap=overlap, blend=blend, batch=batch))
                say("  %s overlap %.2f %-8s batch %d: %3d windows  %7.1f ms per volume  %6.3f Gvox/s  (%.2f ms per window)"
                    % (name, overlap, blend, batch, windows(vol.shape[1:], overlap), t * 1e3, vox / t / 1e9,
                       t * 1e3 / windows(vol.shape[1:], overlap)))
    for k in list(net.__dict__.get("_infer_graphs", {})):
        net._infer_graphs.pop(k)                       # free this volume's captures (and their accumulators)
    torch.cuda.empty_cache()

say("\n== apples to apples: overlap 0 / constant against sliding_window_argmax, 256x512x512 (32 windows)")
for batch in (4, 8):
    ta = timeit(lambda: P.sliding_window_argmax(net, vol256, patch=PATCH, batch=batch))
    tp = timeit(lambda: P.sliding_window_predict(net, vol256, patch=PATCH, overlap=0.0, blend="constant", batch=batch))
    say("  batch %d: sliding_window_argmax %.1f ms, sliding_window_predict %.1f ms (%.3fx)" % (batch, ta * 1e3, tp * 1e3, tp / ta))
net.__dict__.get("_infer_graphs", {}).clear()
torch.cuda.empty_cache()

say("\n== kernels of one eager pass (torch.profiler, batch 4, Gaussian; bytes computed from the shapes)")
KERNELS = ("head_accum_kernel", "window_finalize_kernel", "pack_patches_kernel", "FillFunctor")


def kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: [0.0, 0] for k in KERNELS}
    total = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        if e.device_type is not None and "CUDA" in str(e.device_type):
            total += t
        for k in KERNELS:
            if k in e.key:
                out[k][0] += t * 1e-6
                out[k][1] += e.count
    return out, total * 1e-6


nch, cbt, elt = 4, 2, 2                      # UNetSP: 2 outputs x 2 channels; head input 14 channels = 2 blocks of 8, bf16
for name, vol in (("256x512x512", vol256), ("224x512x512", vol224)):
    vox = vol[0].numel()
    for overlap in (0.0, 0.5):
        nw = windows(vol.shape[1:], overlap)
        ks, tot = kernel_times(lambda: P.sliding_window_predict(net, vol, patch=PATCH, overlap=overlap, blend="gaussian",
                                                                batch=4, graph=False))
        wvox = nw * PATCH ** 3                 # window voxels (all inside the volume at these shapes)
        by = {"head_accum_kernel": wvox * (cbt * 8 * elt + nch * 8),        # head inputs + 64-bit reductions
              "window_finalize_kernel": vox * (nch * 8 + 2 * 4),            # accumulators in, two label volumes out
              "pack_patches_kernel": wvox * (2 * 4 + 8 * elt),              # fp32 volume in, blocked patch out
              "FillFunctor": vox * nch * 8}                                 # the accumulator zeroing (torch.zero_)
        say("  %s overlap %.2f (%d windows): all kernels %.2f ms" % (name, overlap, nw, tot * 1e3))
        for k in KERNELS:
            t, n = ks[k]
            if n:
                say("    %-24s %4d launches %8.3f ms  %6.0f GB/s  (%.0f %% of %.0f GB/s)"
                    % (k, n, t * 1e3, by[k] / t / 1e9, 100 * by[k] / t / 1e9 / HBM_GBS, HBM_GBS))
    net.__dict__.get("_infer_graphs", {}).clear()
    torch.cuda.empty_cache()

if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
