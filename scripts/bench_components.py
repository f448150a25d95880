"""Connected components on one GPU (preprocess.label_components / largest_component, DESIGN.md section 7c).

  volumes   synthetic.head_ct_hu: the 256 x 512 x 512 head CT of scripts/bench_infer.py plus a table slab under the head
            and sparse metal speckle (one large component, one slab, thousands of islands), and the same at 224 x 512 x 512
  timed     hu_threshold -> label_components and hu_threshold -> largest_component at connectivity 6 and 26, and each
            component call alone, with CUDA events after warm-up; the volumes (>= 335 MB of int16 input + >= 470 MB of
            workspace) are larger than the 126 MB L2
  kernels   per-kernel times from torch.profiler in a separate run, with achieved GB/s on algorithmic bytes (labelling:
            mask in + 4 B of labels out per voxel; filter: mask in + mask out) against 6552 GB/s
  scipy     scipy.ndimage.label + numpy.bincount (+ the largest-component selection) on the host cores, the same volume,
            compared bit for bit with the GPU results

    python scripts/bench_components.py [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import torch

import components_oracle as CC
from ctunet_b200 import preprocess as P
from ctunet_b200 import synthetic

HBM_GBS = 6552.0

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None, help="also write the report to this file")
ap.add_argument("--reps", type=int, default=20)
args = ap.parse_args()
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


dev = torch.device("cuda:0")
torch.cuda.set_device(dev)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True)
say("GPU: %s | nvidia-smi: %s | host: %d CPU cores" % (torch.cuda.get_device_name(dev), q.stdout.strip() or "unavailable",
                                                        os.cpu_count()))


def timeit(fn, reps, warm=3):
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


KERNELS = ("ccl_local_kernel", "ccl_boundary_kernel", "ccl_flatten_kernel", "ccl_scan_kernel", "ccl_labels_kernel",
           "ccl_select_kernel", "ccl_filter_kernel")


def kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in KERNELS}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        t = ev.cuda_time_total if t is None else t
        for k in KERNELS:
            if k in ev.key:
                out[k] += t * 1e-6 / 5
    return out


for shape in ((256, 512, 512), (224, 512, 512)):
    hu = synthetic.head_ct_hu(shape, seed=0, device=dev)
    mask = P.hu_threshold(hu, 300)
    vox = mask.numel()
    name = "x".join(map(str, shape))
    say("\n== %s: bone mask (hu >= 300) has %d foreground voxels (%.2f %%)" % (name, int(mask.sum()), 100.0 * float(mask.sum()) / vox))
    m = mask.cpu().numpy()
    for conn in (6, 26):
        lab, cnt = P.label_components(mask, conn)
        big = P.largest_component(mask, conn)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rl, rc = CC.label(m, conn)
        t_label = time.perf_counter() - t0
        t0 = time.perf_counter()
        sizes = np.bincount(rl.ravel(), minlength=int(rc) + 1)
        keep = 1 + int(np.argmax(sizes[1:]))
        rbig = np.where(rl == keep, m, 0).astype(np.uint8)
        t_select = time.perf_counter() - t0
        same_lab = bool(np.array_equal(lab.cpu().numpy(), rl)) and int(cnt) == int(rc)
        same_big = bool(np.array_equal(big.cpu().numpy(), rbig))
        del lab, big
        t_l = timeit(lambda: P.label_components(mask, conn), args.reps)
        t_f = timeit(lambda: P.largest_component(mask, conn), args.reps)
        t_tl = timeit(lambda: P.label_components(P.hu_threshold(hu, 300), conn), args.reps)
        t_tf = timeit(lambda: P.largest_component(P.hu_threshold(hu, 300), conn), args.reps)
        say("  connectivity %d: %d components, largest %d voxels" % (conn, int(rc), int(sizes[keep])))
        say("    label_components    %7.3f ms  (%6.0f GB/s algorithmic: 1 B in + 4 B out per voxel)   hu_threshold -> it: %7.3f ms"
            % (t_l * 1e3, vox * 5 / t_l / 1e9, t_tl * 1e3))
        say("    largest_component   %7.3f ms  (%6.0f GB/s algorithmic: 1 B in + 1 B out per voxel)   hu_threshold -> it: %7.3f ms"
            % (t_f * 1e3, vox * 2 / t_f / 1e9, t_tf * 1e3))
        say("    scipy.ndimage.label %7.1f ms, bincount + select %7.1f ms on the host (%.0fx / %.0fx the GPU)"
            % (t_label * 1e3, t_select * 1e3, t_label / t_l, (t_label + t_select) / t_f))
        say("    GPU == scipy bit for bit: labels + counts %s, largest component %s" % (same_lab, same_big))
        for what, fn, algo in (("label_components", lambda: P.label_components(mask, conn), 5),
                               ("largest_component", lambda: P.largest_component(mask, conn), 2)):
            ks = kernel_times(fn)
            tot = sum(ks.values())
            say("    torch.profiler, %s: kernels %.3f ms = %.0f GB/s of algorithmic bytes (%.0f %% of %.0f GB/s)"
                % (what, tot * 1e3, vox * algo / tot / 1e9, 100 * vox * algo / tot / 1e9 / HBM_GBS, HBM_GBS))
            say("      " + ", ".join("%s %.1f us" % (k, ks[k] * 1e6) for k in KERNELS if ks[k] > 0))
    del hu, mask, m
    torch.cuda.empty_cache()

if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
