"""Cost of floating-point times and of dL/dtimes on one GPU.

A cfg3 EGNO training step (B = 256, N = 20, T = 10, 4 layers: forward + backward), timed with CUDA events in three
arms that alternate: int64 times (nb_egno_forward / nb_egno_backward), the same times as float32 without time gradients
(nb_egno_forward_ft / nb_egno_backward_ft: k_time_table_f for k_time_table), and fractional float32 times that require
grad (one k_time_grad launch more).  Then, in a separate profiled run per arm, the time per launch of the time kernels.

    python tools/float_time_cost.py [--pairs 5] [--steps 20] [--out float_time_cost.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.test_config_space import egno, make_inputs, make_model  # noqa: E402

CASE = egno("egno_cfg3", 101, B=256, N=20, T=10, L=4)
ARMS = ("int64", "float", "float_grad")


def _step_fn(m, inp, arm):
    d = torch.device("cuda:0")
    x0, v0, ea, nodes, lm = (inp[k].to(d) for k in ("x", "v", "ea", "nodes", "lm"))
    edges = [inp["row"].to(d), inp["col"].to(d)]
    t_int = inp["t_out"].to(d)
    t_frac = (t_int.float() + 0.37).contiguous()

    def step():
        x, v = x0.clone().requires_grad_(True), v0.clone().requires_grad_(True)
        t = t_int if arm == "int64" else t_frac.clone().requires_grad_(arm == "float_grad")
        xo, vo, _ = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t)
        (xo.square().mean() + vo.square().mean()).backward()
    return step


def _time(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    agg = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "k_time_" in e.name:
            t, n = agg.get(e.name, (0.0, 0))
            agg[e.name] = (t + e.device_time_total, n + 1)
    return {k: dict(us_per_launch=t / n, launches=n) for k, (t, n) in agg.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    inp = make_inputs(CASE)
    m = make_model(CASE, torch.device("cuda:0"))
    fns = {a: _step_fn(m, inp, a) for a in ARMS}
    for a in ARMS:
        for _ in range(3):
            fns[a]()
    torch.cuda.synchronize()
    ms = {a: [] for a in ARMS}
    for i in range(args.pairs):
        for a in (ARMS if i % 2 == 0 else ARMS[::-1]):
            ms[a].append(_time(fns[a], args.steps))
    res = dict(gpu=smi, case=CASE["name"], steps_per_sample=args.steps,
               arms={a: dict(ms_median=statistics.median(v), ms_min=min(v), ms_max=max(v), kernels=_kernel_times(fns[a]))
                     for a, v in ms.items()})
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
