"""Cost of the input gradients (dL/d node features, edge features, loc_mean) on one GPU.

A cfg3 EGNO training step (B = 256, N = 20, T = 10, 4 layers: forward + backward) and a cfg4-shaped SEGNO step (B = 100,
N = 20, 10 sub-steps), each timed with CUDA events with and without the new gradients requested, the two arms
alternating.  Then, in a separate profiled run, the edge backward kernel's time per launch with and without the EGRAD
instantiation, and the time of the new reduction kernels.

    python tools/input_grad_cost.py [--pairs 5] [--steps 20] [--out input_grad_cost.json]
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

from tests.test_config_space import egno, make_inputs, make_model, segno  # noqa: E402

CASES = [egno("egno_cfg3", 101, B=256, N=20, T=10, L=4), segno("segno_cfg4", 105, B=100, N=20, T=10)]


def _step_fn(c, m, inp, want):
    d = torch.device("cuda:0")
    x0, v0 = inp["x"].to(d), inp["v"].to(d)
    ea0 = inp["ea"].to(d)
    edges = [inp["row"].to(d), inp["col"].to(d)]
    if c["model"] == "egno":
        nodes0, lm0, t_out = inp["nodes"].to(d), inp["lm"].to(d), inp["t_out"].to(d)
    else:
        his0 = inp["his"].to(d)

    def step():
        x, v = x0.clone().requires_grad_(True), v0.clone().requires_grad_(True)
        ea = ea0.clone().requires_grad_(want)
        if c["model"] == "egno":
            nodes, lm = nodes0.clone().requires_grad_(want), lm0.clone().requires_grad_(want)
            xo, vo, ho = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
        else:
            his = his0.clone().requires_grad_(want)
            xo, ho, vo = m(his, x, edges, v, ea, T=c["T"])
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
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name
        if "k_edge_bwd" in name or any(k in name for k in ("k_sum_slices", "k_embed_input_grad", "k_loc_mean_grad",
                                                           "k_sum_over_t")):
            t, n = agg.get(name, (0.0, 0))
            agg[name] = (t + e.device_time_total, n + 1)
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
    res = dict(gpu=smi, cases={})
    for c in CASES:
        inp = make_inputs(c)
        m = make_model(c, torch.device("cuda:0"))
        fns = {w: _step_fn(c, m, inp, w) for w in (False, True)}
        for w in (False, True):
            for _ in range(3):
                fns[w]()
        torch.cuda.synchronize()
        ms = {False: [], True: []}
        for _ in range(args.pairs):
            for w in (False, True):
                ms[w].append(_time(fns[w], args.steps))
        r = {("with" if w else "without"): dict(ms_median=statistics.median(v), ms_min=min(v), ms_max=max(v))
             for w, v in ms.items()}
        r["kernels_without"] = _kernel_times(fns[False])
        r["kernels_with"] = _kernel_times(fns[True])
        res["cases"][c["name"]] = r
        print(c["name"], json.dumps(r, indent=1))
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
