"""Cost of Dropout3d on the fused path (GPU): the captured training step (TrainStep(graph=True), bf16, batch 4 x 128^3) of
UNetSP and recAE_v2_fixed with dropout_p = 0 and 0.1 on every site, the two arms alternating in one process, and the
BatchNorm+ReLU(+MaxPool) kernels alone at 7 channels, 4 x 128^3, with and without keep factors.
    python scripts/bench_dropout.py [--steps 20 --rounds 5]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch

import ctunet_b200 as C
from ctunet_b200 import _lib
from ctunet_b200._lib import CTU_BF16, call, stream_ptr
from ctunet_b200.synthetic import make_training_batch
from ctunet_b200.trainer import TrainStep
from bench_kernels_common import act, timeit   # noqa: E402  (same directory)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return out or torch.cuda.get_device_name(0)


def time_steps(step, x, t, steps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        step(x, t)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps


def bench_model(name, cin, handler, batch, size, steps, rounds, arms):
    x, t = make_training_batch(batch, cin, size, seed=3)
    if handler == "single":
        t = t[0]
    runs = {}
    for p in arms:
        torch.manual_seed(0)
        net = getattr(C, name)().cuda()
        for _, m, _ in net._dropout_sites():
            m.p = p
        step = TrainStep(net, handler, lr=1e-4, graph=True)
        for _ in range(5):                      # warm-up + capture
            step(x, t)
        torch.cuda.synchronize()
        runs[p] = (net, step)
    ms = {p: [] for p in arms}
    for _ in range(rounds):
        for p in arms:                          # alternating arms: drifts of the shared machine hit both
            ms[p].append(time_steps(runs[p][1], x, t, steps))
    res = {"model": name, "batch": batch, "size": size, "steps_per_round": steps, "rounds": rounds}
    for p in arms:
        res["p=%g" % p] = {"ms_per_step_median": float(np.median(ms[p])), "ms_per_step_min": float(np.min(ms[p])),
                           "ms_per_step_max": float(np.max(ms[p])), "launches_per_step": runs[p][1].launches_per_step}
    base = res["p=%g" % arms[0]]["ms_per_step_median"]
    for p in arms[1:]:
        res["p=%g_over_p=%g" % (p, arms[0])] = res["p=%g" % p]["ms_per_step_median"] / base
    del runs
    torch.cuda.empty_cache()
    return res


def bench_bn(n=4, c=7, s=128):
    """The BatchNorm kernels of one dropout site alone: forward (plain and pooled), backward reduce + apply."""
    cpad = (c + 7) // 8 * 8
    y, a, dA = act(n, c, s, s, s), act(n, c, s, s, s), act(n, c, s, s, s)
    pooled, dP = act(n, c, s // 2, s // 2, s // 2), act(n, c, s // 2, s // 2, s // 2)
    dy = act(n, c, s, s, s)
    ss = torch.cat([torch.rand(cpad, device="cuda") + 0.5, torch.randn(cpad, device="cuda") * 0.1,
                    torch.zeros(cpad, device="cuda"), torch.ones(cpad, device="cuda")])
    gamma = torch.ones(cpad, device="cuda")
    sums2 = torch.zeros(2 * cpad, dtype=torch.float64, device="cuda")
    dg, db = torch.empty(cpad, device="cuda"), torch.empty(cpad, device="cuda")
    keep = ((torch.rand(n, cpad, device="cuda") > 0.1).float() / 0.9).contiguous()
    count = float(n * s ** 3)
    out = {"n": n, "c": c, "size": s}
    for tag, k in (("plain", None), ("keep", keep.data_ptr())):
        sfx = "_drop" if k is not None else ""
        ex = (k,) if k is not None else ()
        for pool in (False, True):
            pp = pooled.data_ptr() if pool else None
            pd = dP.data_ptr() if pool else None
            t_fwd = timeit(lambda: call("ctu_bn_relu_fwd" + sfx, CTU_BF16, y.data_ptr(), ss.data_ptr(), a.data_ptr(), pp,
                                        c, n, s, s, s, 0, *ex, stream_ptr()))
            t_red = timeit(lambda: call("ctu_bn_relu_bwd_reduce" + sfx, CTU_BF16, y.data_ptr(), ss.data_ptr(), dA.data_ptr(),
                                        pd, sums2.data_ptr(), c, n, s, s, s, 0, *ex, stream_ptr()))
            t_app = timeit(lambda: call("ctu_bn_relu_bwd_apply" + sfx, CTU_BF16, y.data_ptr(), ss.data_ptr(),
                                        gamma.data_ptr(), dA.data_ptr(), pd, sums2.data_ptr(), count, dy.data_ptr(),
                                        dg.data_ptr(), db.data_ptr(), c, n, s, s, s, 0, *ex, stream_ptr()))
            out["%s_%s_us" % (tag, "pooled" if pool else "unpooled")] = {"fwd": round(t_fwd, 1), "bwd_reduce": round(t_red, 1),
                                                                          "bwd_apply": round(t_app, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--batch", type=int, default=4)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    print(json.dumps({"gpu": info}))
    arms = (0.0, 0.1)
    for name, cin, handler in (("UNetSP", 2, "double"), ("recAE_v2_fixed", 1, "single")):
        res = bench_model(name, cin, handler, args.batch, args.size, args.steps, args.rounds, arms)
        res["gpu"] = info
        print(json.dumps(res))
    res = bench_bn()
    res["gpu"] = info
    print(json.dumps(res))


if __name__ == "__main__":
    main()
