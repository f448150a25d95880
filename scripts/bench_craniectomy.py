"""Cost of the virtual craniectomy on the device (GPU): at batch 4 x 128^3 with the atlas channel,
  1. the draw (ctu_craniectomy_draw: per-chunk bone counts + the single-CTA draw), the fused encoder
     ctu_craniectomy_encode_flaprec without and with RandomAffine matrices, against the plain encoders
     (ctu_encode_flaprec_bits / _u8) that take three ready masks, in bits and uint8 formats, CUDA events over many calls
     replayed from a graph;
  2. the captured UNetSP bf16 step via step_from_skull_bits against step_from_bits fed ready masks, the two arms
     alternating in one process, median of rounds x steps, and the per-kernel device times of one craniectomy step;
  3. for scale, the wall time per batch of the earlier routes: SkullRandomHole on the device (host-RNG draws, one
     count_nonzero sync per sample) then step_from_masks, and the reference's numpy blank_patch on the host cores.
    python scripts/bench_craniectomy.py [--steps 20 --rounds 5 --out profiles/r3_bench_craniectomy.txt]"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch

import ctunet_b200 as C
from ctunet_b200._lib import call, stream_ptr
from ctunet_b200.trainer import TrainStep
from ctunet_b200.utilities import pack_mask_bits, radius_bounds
from ctunet_b200.synthetic import make_training_batch
from bench_kernels_common import timeit   # noqa: E402  (same directory)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return out or torch.cuda.get_device_name(0)


def kernels(full, full_bits, masks, bits, atlas, vol, reps):
    b = full.shape[0]
    d, h, w = vol
    s = d * h * w
    image = torch.empty((b, 2) + vol, device="cuda")
    fm = torch.empty((b,) + vol, dtype=torch.uint8, device="cuda")
    lm = torch.empty_like(fm)
    rc, ra = C.RandomCraniectomy(), C.RandomAffine()
    params = rc.draw(full)
    _, mats = ra.draw(b, vol, "cuda")
    key, counter = rc._state[full.device]
    min_r, max_r = (int(r) for r in radius_bounds(vol))
    nbytes = C._lib.load().ctu_craniectomy_workspace_bytes(b, d, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = {"params_shapes": params[:, 1].tolist(), "params_radius": params[:, 2].tolist()}
    wbytes = b * s * (8 + 2)       # float image with atlas channel (8 B/voxel) + two uint8 label masks (2 B/voxel)
    for fmt, flag, src in (("bits", 1, full_bits), ("u8", 0, full)):
        res = {}
        draw = lambda: call("ctu_craniectomy_draw", flag, src.data_ptr(), b, d, h, w, 1.0, 7, min_r, max_r, key,   # noqa: E731
                            counter.data_ptr(), params.data_ptr(), ws.data_ptr(), nbytes, stream_ptr())
        res["draw_us"] = round(timeit(draw, reps), 2)
        rc.draw(full)                                        # the holes every encoder call below cuts
        for tag, m in (("hole", None), ("hole_affine", mats)):
            us = timeit(lambda: call("ctu_craniectomy_encode_flaprec", flag, src.data_ptr(), params.data_ptr(),
                                     atlas.data_ptr(), m.data_ptr() if m is not None else None, image.data_ptr(),
                                     fm.data_ptr(), lm.data_ptr(), b, 2, d, h, w, stream_ptr()), reps)
            res["%s_us" % tag] = round(us, 1)
            res["%s_write_GBps" % tag] = round(wbytes / us / 1e3, 1)
        if fmt == "bits":
            us = timeit(lambda: call("ctu_encode_flaprec_bits", *[t.data_ptr() for t in bits], atlas.data_ptr(),
                                     image.data_ptr(), fm.data_ptr(), lm.data_ptr(), b, 2, s, stream_ptr()), reps)
            res["plain_encode_flaprec_bits_us"] = round(us, 1)
        else:
            def plain_step_input():                          # what step_from_masks runs: image encoder + two mask copies
                call("ctu_encode_flaprec_u8", *[t.data_ptr() for t in masks], atlas.data_ptr(), image.data_ptr(), None,
                     None, b, 2, s, stream_ptr())
                fm.copy_(masks[1], non_blocking=True)
                lm.copy_(masks[2], non_blocking=True)
            res["plain_encode_flaprec_u8_plus_mask_copies_us"] = round(timeit(plain_step_input, reps), 1)
        plain = res.get("plain_encode_flaprec_bits_us") or res["plain_encode_flaprec_u8_plus_mask_copies_us"]
        res["plain_write_GBps"] = round(wbytes / plain / 1e3, 1)
        res["hole_over_plain"] = round(res["hole_us"] / plain, 3)
        res["hole_affine_over_plain"] = round(res["hole_affine_us"] / plain, 3)
        out[fmt] = res
    out["write_bytes_per_call"] = wbytes
    return out


def time_steps(fn, steps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps


def profile_kernels(fn, n, match):
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
        agg = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA":
                t = agg.setdefault(ev.name, [0, 0.0])
                t[0] += 1
                t[1] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        return {"device_us_per_step_total": round(sum(v[1] for v in agg.values()) / n, 1),
                "kernels_us": {k[:110]: round(v[1] / v[0], 1) for k, v in agg.items() if any(m in k for m in match)}}
    except Exception as e:                                   # the timing above stands on its own
        return {"error": repr(e)}


def step_bench(full_bits, bits, atlas, vol, steps, rounds):
    runs = {}
    for arm in ("plain", "craniectomy"):
        torch.manual_seed(0)
        net = C.UNetSP().cuda().train()
        if arm == "plain":
            step = TrainStep(net, "double", lr=1e-4, graph=True)
            fn = (lambda step=step: step.step_from_bits(*bits, vol, atlas))
        else:
            step = TrainStep(net, "double", lr=1e-4, graph=True, craniectomy=C.RandomCraniectomy())
            fn = (lambda step=step: step.step_from_skull_bits(full_bits, vol, atlas))
        for _ in range(5):                       # warm-up + capture
            fn()
        torch.cuda.synchronize()
        runs[arm] = (step, fn)
    ms = {arm: [] for arm in runs}
    for _ in range(rounds):
        for arm in runs:                         # alternating arms: drifts of the shared machine hit both
            ms[arm].append(time_steps(runs[arm][1], steps))
    res = {"model": "UNetSP", "dtype": "bf16", "batch": full_bits.shape[0], "size": vol, "steps_per_round": steps,
           "rounds": rounds}
    for arm in runs:
        res[arm] = {"ms_per_step_median": round(float(np.median(ms[arm])), 4),
                    "ms_per_step_min": round(float(np.min(ms[arm])), 4), "ms_per_step_max": round(float(np.max(ms[arm])), 4),
                    "launches_per_step": runs[arm][0].launches_per_step}
    res["craniectomy_over_plain"] = round(res["craniectomy"]["ms_per_step_median"] / res["plain"]["ms_per_step_median"], 4)
    res["profile_craniectomy_step"] = profile_kernels(runs["craniectomy"][1], 3, ("craniectomy", "affine_gather"))
    del runs
    torch.cuda.empty_cache()
    return res


def earlier_routes(full, atlas, steps):
    """Wall time per batch: SkullRandomHole on the device (host RNGs, a count_nonzero sync per sample, a launch chain per
    sample) then the captured step_from_masks; and the reference's numpy blank_patch on the host (random_blank_patch
    with its host draws, transforms.py:241-300, as oracle/unet_oracle.py restates it)."""
    from oracle import unet_oracle as O
    torch.manual_seed(0)
    step = TrainStep(C.UNetSP().cuda().train(), "double", lr=1e-4, graph=True)
    hole = C.SkullRandomHole(double_output=True)

    def one():
        s = hole({"image": full})
        return step.step_from_masks(s["image"], s["target"][0], s["target"][1], atlas)
    for _ in range(4):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    dev_ms = (time.perf_counter() - t0) / steps * 1e3
    t0 = time.perf_counter()
    for _ in range(steps):
        hole({"image": full})
    torch.cuda.synchronize()
    hole_ms = (time.perf_counter() - t0) / steps * 1e3
    host = full.cpu().numpy()
    np.random.seed(0)
    random.seed(0)
    t0 = time.perf_counter()
    for b in range(host.shape[0]):
        vol = host[b]
        idx = np.argwhere(vol > 0)
        centre = idx[np.random.choice(len(idx))]
        lo, hi = O.radius_bounds(vol.shape)
        size = np.random.randint(lo, hi)
        shape = ("sphere", "box", "flap")[np.random.randint(0, 3)]
        O.blank_patch(vol, centre, size, shape)
    host_ms = (time.perf_counter() - t0) * 1e3
    return {"skull_random_hole_device_then_step_from_masks_ms_per_batch": round(dev_ms, 3),
            "skull_random_hole_device_alone_ms_per_batch": round(hole_ms, 3),
            "reference_numpy_blank_patch_host_ms_per_batch": round(host_ms, 1), "host_threads": os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_craniectomy.txt"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    C.set_compute_dtype("bf16")
    lines = []

    def emit(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        lines.append(s)

    info = gpu_info()
    emit({"gpu": info})
    img, (sk_t, fl_t) = make_training_batch(4, 2, 128, seed=3)
    masks = [t.to(torch.uint8).contiguous() for t in (img[:, 0], sk_t[:, 1], fl_t[:, 1])]
    bits = [pack_mask_bits(m) for m in masks]
    full, full_bits = masks[1], bits[1]
    atlas = img[0, 1].contiguous()
    vol = tuple(full.shape[1:])
    for res in (kernels(full, full_bits, masks, bits, atlas, vol, args.reps),
                step_bench(full_bits, bits, atlas, vol, args.steps, args.rounds),
                earlier_routes(full, atlas, args.steps)):
        res["gpu"] = info
        emit(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# scripts/bench_craniectomy.py --steps %d --rounds %d --reps %d\n" % (args.steps, args.rounds, args.reps))
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
