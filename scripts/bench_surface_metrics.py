"""Surface-distance evaluation on one GPU (utilities.surface_metrics, DESIGN.md section 7d).

  inputs    the skull (largest component of the thresholded synthetic.head_ct_hu) against a copy shifted by (2, -3, 1)
            voxels with added one-voxel islands, at 256 x 512 x 512 and 224 x 512 x 512; and a 4 x 128^3 batch of skull
            phantoms against phantoms of other seeds (the size of a validation batch of training).  Each without spacing
            (voxel units) and with spacing (1.25, 0.5, 0.5) mm.  The volumes and workspaces are larger than the 126 MB L2
            except the 128^3 batch, which is reported as it is.
  timed     one surface_metrics call (percentile 95, tolerance 1), CUDA events over --reps calls after warm-up
  kernels   per-kernel times from torch.profiler in a separate pass, with achieved GB/s on the algorithmic bytes: both
            masks in, per set the edge flags written once and read twice (pass 1 and the partner read of pass 3), and
            the distance planes once per pass (written by pass 1, read and written by pass 2, read by pass 3); the key
            list and the selection are left out of the count
  scipy     tests/surface_oracle.py (binary_erosion, distance_transform_edt, numpy.percentile / mean) on the host cores,
            the same inputs, compared with the GPU: bit for bit without spacing (assd to relative 1e-12), to relative
            1e-12 with spacing

    python scripts/bench_surface_metrics.py [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import surface_oracle as SO
from ctunet_b200 import preprocess as P
from ctunet_b200 import synthetic
from ctunet_b200.utilities import surface_metrics

HBM_GBS = 6552.0
SPACING = (1.25, 0.5, 0.5)

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


KERNELS = ("mask_edges_kernel", "edt_row_kernel", "edt_axis_kernel", "pct_rank_kernel", "radix_hist_kernel",
           "radix_pick_kernel", "surface_finalize_kernel")


def kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        t = ev.cuda_time_total if t is None else t
        for k in KERNELS:
            if k in ev.key:
                name = ev.key.split("(")[0].replace("void ", "").replace("ctu::", "")
                out[name] = out.get(name, 0.0) + t * 1e-6 / 5
    return out


def skull_pair(shape):
    skull = P.largest_component(P.hu_threshold(synthetic.head_ct_hu(shape, seed=0, device=dev), 300))
    moved = torch.zeros_like(skull)
    moved[2:, :-3, 1:] = skull[:-2, 3:, :-1]
    g = torch.Generator(device=dev).manual_seed(1)
    moved[torch.rand(shape, device=dev, generator=g) < 1e-5] = 1
    return skull, moved


def phantom_batch():
    p = torch.stack([synthetic.skull_phantom(128, s, dev) for s in range(4)])
    t = torch.stack([synthetic.skull_phantom(128, 100 + s, dev) for s in range(4)])
    return p, t


def matches(got, ref, weighted):
    for k in SO.KEYS:
        g, r = np.atleast_1d(got[k].cpu().numpy()), np.atleast_1d(np.asarray(ref[k]))
        fin = np.isfinite(r)
        if not np.array_equal(g[~fin], r[~fin], equal_nan=True) or not np.array_equal(np.isfinite(g), fin):
            return False
        if k == "assd" or (weighted and k in ("hausdorff", "hausdorff_percentile")):
            if not np.allclose(g[fin], r[fin], rtol=1e-12, atol=0):
                return False
        elif not np.array_equal(g[fin], r[fin]):
            return False
    return True


all_ok = True
for name, make in (("256x512x512 skull pair", lambda: skull_pair((256, 512, 512))),
                   ("224x512x512 skull pair", lambda: skull_pair((224, 512, 512))),
                   ("4x128^3 phantom batch", phantom_batch)):
    p, t = make()
    pn, tn = p.cpu().numpy(), t.cpu().numpy()
    vox = p.numel()
    say("\n== %s: |P| = %d, |T| = %d voxels" % (name, int(p.sum()), int(t.sum())))
    for sp in (None, SPACING):
        kw = dict(spacing=sp, percentile=95.0, tolerance=1.0)
        got = surface_metrics(p, t, **kw)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ref = SO.surface_metrics(pn, tn, **kw)
        t_cpu = time.perf_counter() - t0
        ok = matches(got, ref, sp is not None)
        all_ok &= ok
        t_gpu = timeit(lambda: surface_metrics(p, t, **kw), args.reps)
        plane = 8 if sp is not None else 4
        algo = 2 * vox + 2 * vox * (3 + 4 * plane)
        label = "voxel units" if sp is None else "spacing %s" % (SPACING,)
        vals = ", ".join("%s %s" % (k, np.array2string(np.atleast_1d(got[k].cpu().numpy()), precision=6)) for k in SO.KEYS)
        say("  %s: %.3f ms per call (%d calls, CUDA events), %.0f GB/s of algorithmic bytes (%.2f GB)"
            % (label, t_gpu * 1e3, args.reps, algo / t_gpu / 1e9, algo / 1e9))
        say("    %s" % vals)
        say("    scipy oracle on the host: %.2f s (%.0fx the GPU); GPU == oracle: %s" % (t_cpu, t_cpu / t_gpu, ok))
        ks = kernel_times(lambda: surface_metrics(p, t, **kw))
        tot = sum(ks.values())
        say("    torch.profiler: kernels %.3f ms = %.0f GB/s of algorithmic bytes (%.0f %% of %.0f GB/s)"
            % (tot * 1e3, algo / tot / 1e9, 100 * algo / tot / 1e9 / HBM_GBS, HBM_GBS))
        say("      " + ", ".join("%s %.1f us" % (k, v * 1e6) for k, v in sorted(ks.items(), key=lambda kv: -kv[1])))
    del p, t, pn, tn
    torch.cuda.empty_cache()

say("\nevery GPU value equals the oracle (bit for bit without spacing, assd to 1e-12; 1e-12 with spacing): %s" % all_ok)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
