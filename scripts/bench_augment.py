"""Cost of the random affine augmentation (GPU): at batch 4 x 128^3,
  1. the fused encoder ctu_affine_encode_flaprec with random draws and with the identity, against the plain encoders
     (ctu_encode_flaprec_bits / _u8), in bits and uint8 formats, CUDA events over many calls, with the achieved write
     bandwidth against the device copy bandwidth, and the draw launch alone;
  2. the captured UNetSP bf16 step_from_bits with and without augmentation, the two arms alternating in one process,
     median of rounds x steps, and the per-kernel device times of one augmenting step (torch.profiler);
  3. scipy.ndimage.affine_transform(order=0) of the same three masks x 4 samples on the host cores.
    python scripts/bench_augment.py [--steps 20 --rounds 5 --out profiles/r3_bench_augment.txt]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch

import ctunet_b200 as C
from ctunet_b200 import _lib
from ctunet_b200._lib import call, stream_ptr
from ctunet_b200.trainer import TrainStep
from ctunet_b200.utilities import pack_mask_bits
from ctunet_b200.synthetic import make_training_batch
from bench_kernels_common import timeit   # noqa: E402  (same directory)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return out or torch.cuda.get_device_name(0)


def copy_bandwidth():
    """Device-to-device copy of 2 GiB (larger than L2): bytes read + written per second."""
    a = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    us = timeit(lambda: b.copy_(a), reps=10)
    return 2 * a.numel() / us / 1e3          # GB/s


def kernels(masks, bits, atlas, vol, reps):
    b = masks[0].shape[0]
    d, h, w = vol
    s = d * h * w
    image = torch.empty((b, 2) + vol, device="cuda")
    fm = torch.empty((b,) + vol, dtype=torch.uint8, device="cuda")
    lm = torch.empty_like(fm)
    ra = C.RandomAffine()
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    params = torch.empty(b, 10, device="cuda")
    rnd = torch.empty(b, 3, 4, device="cuda")
    rng = (_lib.c_float * 8)(*ra._ranges)
    draw = lambda: call("ctu_affine_draw", b, d, h, w, rng, ra._flip_axes, 1234, counter.data_ptr(),   # noqa: E731
                        params.data_ptr(), rnd.data_ptr(), stream_ptr())
    draw()
    eye = torch.eye(3, 4, device="cuda").repeat(b, 1, 1).contiguous()
    out = {"draw_us": round(timeit(draw, reps), 2)}
    # bytes the encoders must write: float image with atlas channel (8 B/voxel) + two uint8 label masks (2 B/voxel)
    wbytes = b * s * (8 + 2)
    for fmt, srcs in (("bits", bits), ("u8", masks)):
        flag = 1 if fmt == "bits" else 0
        res = {}
        for tag, mats in (("random", rnd), ("identity", eye)):
            us = timeit(lambda: call("ctu_affine_encode_flaprec", flag, *[t.data_ptr() for t in srcs], atlas.data_ptr(),
                                     mats.data_ptr(), image.data_ptr(), fm.data_ptr(), lm.data_ptr(), b, 2, d, h, w,
                                     stream_ptr()), reps)
            res["affine_%s_us" % tag] = round(us, 1)
            res["affine_%s_write_GBps" % tag] = round(wbytes / us / 1e3, 1)
        if fmt == "bits":
            us = timeit(lambda: call("ctu_encode_flaprec_bits", *[t.data_ptr() for t in bits], atlas.data_ptr(),
                                     image.data_ptr(), fm.data_ptr(), lm.data_ptr(), b, 2, s, stream_ptr()), reps)
            res["plain_encode_flaprec_bits_us"] = round(us, 1)
        else:
            # what step_from_masks runs today: the image-only encoder, then the two label masks copied into the step's
            # static inputs
            us = timeit(lambda: call("ctu_encode_flaprec_u8", *[t.data_ptr() for t in masks], atlas.data_ptr(),
                                     image.data_ptr(), None, None, b, 2, s, stream_ptr()), reps)
            res["plain_encode_flaprec_u8_image_only_us"] = round(us, 1)

            def plain_step_input():
                call("ctu_encode_flaprec_u8", *[t.data_ptr() for t in masks], atlas.data_ptr(), image.data_ptr(), None,
                     None, b, 2, s, stream_ptr())
                fm.copy_(masks[1], non_blocking=True)
                lm.copy_(masks[2], non_blocking=True)
            us = timeit(plain_step_input, reps)
            res["plain_encode_flaprec_u8_plus_mask_copies_us"] = round(us, 1)
        plain = res.get("plain_encode_flaprec_bits_us") or res["plain_encode_flaprec_u8_plus_mask_copies_us"]
        res["plain_write_GBps"] = round(wbytes / plain / 1e3, 1)
        res["affine_random_over_plain"] = round(res["affine_random_us"] / plain, 3)
        res["affine_identity_over_plain"] = round(res["affine_identity_us"] / plain, 3)
        out[fmt] = res
    out["write_bytes_per_call"] = wbytes
    return out, rnd


def time_steps(fn, steps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps


def step_bench(bits, atlas, vol, steps, rounds, out_dir):
    runs = {}
    for arm in ("plain", "augment"):
        torch.manual_seed(0)
        net = C.UNetSP().cuda().train()
        step = TrainStep(net, "double", lr=1e-4, graph=True, augment=C.RandomAffine() if arm == "augment" else None)
        fn = (lambda step=step: step.step_from_bits(*bits, vol, atlas))
        for _ in range(5):                       # warm-up + capture
            fn()
        torch.cuda.synchronize()
        runs[arm] = (step, fn)
    ms = {arm: [] for arm in runs}
    for _ in range(rounds):
        for arm in runs:                         # alternating arms: drifts of the shared machine hit both
            ms[arm].append(time_steps(runs[arm][1], steps))
    res = {"model": "UNetSP", "dtype": "bf16", "batch": bits[0].shape[0], "size": vol, "steps_per_round": steps,
           "rounds": rounds}
    for arm in runs:
        res[arm] = {"ms_per_step_median": round(float(np.median(ms[arm])), 4), "ms_per_step_min": round(float(np.min(ms[arm])), 4),
                    "ms_per_step_max": round(float(np.max(ms[arm])), 4), "launches_per_step": runs[arm][0].launches_per_step}
    res["augment_over_plain"] = round(res["augment"]["ms_per_step_median"] / res["plain"]["ms_per_step_median"], 4)
    # per-kernel device times of 3 augmenting steps (a separate, profiled run)
    prof_tbl = None
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                runs["augment"][1]()
            torch.cuda.synchronize()
        agg = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA":
                t = agg.setdefault(ev.name, [0, 0.0])
                t[0] += 1
                t[1] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        top = sorted(agg.items(), key=lambda kv: -kv[1][1])
        total = sum(v[1] for _, v in top)
        prof_tbl = {"device_us_per_step_total": round(total / 3, 1),
                    "affine": {k: round(v[1] / v[0], 1) for k, v in top if "affine" in k},
                    "top10_us_per_step": [(k[:80], round(v[1] / 3, 1)) for k, v in top[:10]]}
    except Exception as e:                       # the timing above stands on its own
        prof_tbl = {"error": repr(e)}
    res["profile_augmenting_step"] = prof_tbl
    del runs
    torch.cuda.empty_cache()
    return res


def scipy_bench(masks, mats):
    """scipy.ndimage.affine_transform(order=0) of the three masks of every sample with the same maps (output coordinate
    -> input coordinate, as here), on the host; and how many voxels agree with the GPU gather (scipy rounds the
    coordinate its own way, so a few voxels on rounding ties differ)."""
    from scipy import ndimage
    host = [m.cpu().numpy() for m in masks]
    M = mats.cpu().numpy().astype(np.float64)
    t0 = time.perf_counter()
    out = [np.empty_like(h) for h in host]
    for b in range(host[0].shape[0]):
        for h, o in zip(host, out):
            o[b] = ndimage.affine_transform(h[b], M[b, :, :3], offset=M[b, :, 3], order=0, mode="constant", cval=0)
    sec = time.perf_counter() - t0
    gpu = [t.cpu().numpy() for t in C.affine_masks(list(masks), mats)]
    agree = float(np.mean([np.mean(a == g) for a, g in zip(out, gpu)]))
    return {"seconds_3_masks_x_%d_samples" % host[0].shape[0]: round(sec, 3), "threads": os.cpu_count(),
            "voxel_agreement_with_gpu": round(agree, 6)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r3_bench_augment.txt"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
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
    atlas = img[0, 1].contiguous()
    vol = tuple(masks[0].shape[1:])
    emit({"copy_GBps_read_plus_write": round(copy_bandwidth(), 1), "gpu": info})
    res, mats = kernels(masks, bits, atlas, vol, args.reps)
    res["gpu"] = info
    emit(res)
    res = step_bench(bits, atlas, vol, args.steps, args.rounds, None)
    res["gpu"] = info
    emit(res)
    res = scipy_bench(masks, mats)
    res["gpu"] = info
    emit(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# scripts/bench_augment.py --steps %d --rounds %d --reps %d\n" % (args.steps, args.rounds, args.reps))
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
