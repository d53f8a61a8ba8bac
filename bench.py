#!/usr/bin/env python
"""bench.py — throughput of the EGNO / SEGNO hot path on B200 (BASELINE.json metric: trajectories/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                   # + the last timed step's results as DIR/<name>.npy
    python bench.py --impl reference --gpus N ...            # the reference's CPU implementation (oracle port)
    torchrun --nproc-per-node N bench.py --gpus N ...        # one rank per GPU (weak scaling: B per GPU fixed)

A "step" is one training pass (forward + MSE loss + backward + Adam) of the 20-body EGNO (BASELINE.json
configs[2]: N=20, num_timesteps=10, hidden 64, 4 layers) over one batch of B=256 synthetic trajectories
(main.py:32 default batch) per GPU.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import functools
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

_STDOUT_FD = None


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _STDOUT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_STDOUT_FD, data)


METRIC = "train trajectories/s (EGNO 20-body, fwd+bwd+Adam)"
UNIT = "trajectories/s"

# per-edge MACs of the reference formulas (SURVEY.md §8): phi_e = 131*64 + 64*64, phi_x = 64*64 + 64
MAC_EDGE_REF = 131 * 64 + 64 * 64 + 64 * 64 + 64
# MACs the fused edge kernel itself executes per edge (first layer's h-part runs per node, outside it)
MAC_EDGE_KERNEL = 64 * 64 + 64 * 64 + 64 + 3 * 64
DUMP_BYTES = 64 << 20      # --dump-outputs: upper bound of the files written


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="timed training steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="trajectories per GPU per step")
    ap.add_argument("--n-balls", type=int, default=20)
    ap.add_argument("--timesteps", type=int, default=10)
    ap.add_argument("--layers", type=int, default=4)
    ap.add_argument("--cpu-sample", type=int, default=32, help="trajectories per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the SEGNO / inference side numbers")
    ap.add_argument("--quick", action="store_true", help="device-resident timing only (for profiler runs)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying one CUDA "
                                                            "graph per training step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as "
                    "DIR/<name>.npy (float32): loss, x_out, v_out, h_out (the model's outputs), grads and params (after the "
                    "optimizer step), both flat in named_parameters() order; rows are sampled with a fixed seed to keep "
                    f"the files within {DUMP_BYTES >> 20} MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of this repo's CUDA path (--impl ours)")
    return args


def dump_outputs(outdir, arrays):
    """Each array -> <outdir>/<name>.npy in float32.  When the arrays together exceed DUMP_BYTES, every array keeps the
    same share of its rows, drawn by a generator seeded with 0, so two runs of the same arguments keep the same rows."""
    os.makedirs(outdir, exist_ok=True)
    total = sum(4 * a.numel() for a in arrays.values())
    room = DUMP_BYTES - 4096 * len(arrays)         # less the .npy headers
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if total > room and a.dim() > 0:
            keep = a.shape[0] * room // total
            a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
        np.save(os.path.join(outdir, name + ".npy"), a.numpy())


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, window=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines
        scope = "whole run (sampler start to stop)"
        if window is not None:
            inside = [x for x in lines if window[0] <= x[0] <= window[1] + 0.05]
            if inside:
                lines, scope = inside, "timed region"
            else:
                scope = "warm-up + timed region (timed region shorter than one sampling period)"
        for _, ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


# ------------------------------------------------------------------------------------------------ CPU arm
def _reference_or_port():
    """The reference's own modules when the unmodified copy is installed (oracle/_ref, made by oracle/make_ref.py in the
    build container; it travels to the GPU box), else None (the oracle port is timed instead)."""
    try:
        from oracle import ref_loader as RL

        if RL.reference_available():
            return RL.load_reference(), RL
    except Exception as e:       # a broken install must not take the bench down: fall back to the port and say so
        print(f"reference import failed ({e}); timing the oracle port", file=sys.stderr)
    return None, None


def cpu_reference_arm(args, steps, warmup, sample, model="egno", device="cpu"):
    """The reference's implementation of the path on the host cores: the reference's real `EGNO` / `SEGNO` modules
    (kind "reference") when oracle/_ref is installed, else the oracle port (kind "port"); forward + the callers' MSE +
    backward + torch.optim.Adam with all host threads, on a bounded sample of the workload.  With device="cuda" the
    oracle port runs the same PyTorch eager ops on the B200 (same-GPU context for the hand-written kernels)."""
    from oracle import nbody_oracle as O
    from no_node_comparison_b200 import synth

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    N, T, L = args.n_balls, args.timesteps, args.layers
    R, RL = _reference_or_port() if device == "cpu" else (None, None)
    torch.manual_seed(1)
    dev = torch.device(device)
    row, col = synth.canonical_edges(sample, N)
    if model == "egno":
        s = synth.sample_state("charged", sample, N, seed=0)
        x, nodes, ea, v, lm = synth.egno_features(s["loc"], s["vel"], s["charges"], row, col)
        t_out = torch.arange(1, T + 1)[None].repeat(sample, 1)
        target = x.repeat(T, 1) + 0.05 * torch.randn(T * sample * N, 3, generator=torch.Generator().manual_seed(1))
        x, nodes, ea, v, lm, t_out, target, row, col = (t.to(dev) for t in (x, nodes, ea, v, lm, t_out, target, row, col))
        if R is not None:
            m = R.EGNO(n_layers=L, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T,
                       device="cpu")
            params = list(m.parameters())
            fwd = lambda: m(x, nodes, [row, col], ea, v=v, loc_mean=lm, timesteps_out=t_out)[0]
        else:
            import no_node_comparison_b200 as nb

            holder = nb.EGNO(n_layers=L, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2,
                             num_timesteps=T, device="cpu")
            p = {k: t.detach().clone().to(dev).requires_grad_(True) for k, t in holder.state_dict().items()}
            params = list(p.values())
            fwd = lambda: O.egno_forward(p, x, nodes, row, col, ea, v, lm, t_out, n_layers=L, num_timesteps=T)[0]
        opt = torch.optim.Adam(params, lr=1e-4, weight_decay=1e-8)
        what = f"EGNO N={N}, T={T}, L={L}"
    else:
        s = synth.sample_state("gravity", sample, N, seed=0)
        his, x, v, ea = synth.segno_features(s["loc"], s["vel"], s["charges"], row, col)
        target = x + 0.05 * torch.randn(sample * N, 3, generator=torch.Generator().manual_seed(1))
        his, x, v, ea, target, row, col = (t.to(dev) for t in (his, x, v, ea, target, row, col))
        if R is not None:
            m = R.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", n_layers=8, recurrent=True)
            params = [q for k, q in m.named_parameters()]
            # SEGNO.forward at reference HEAD returns its inputs (SURVEY.md 0); the semantics its callers assume:
            fwd = lambda: m.forward_step(m.embedding(his), x, [row, col], v, ea, T=T)[0]
        else:
            import no_node_comparison_b200 as nb

            holder = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", n_layers=8, recurrent=True)
            p = {k: t.detach().clone().to(dev).requires_grad_(True) for k, t in holder.state_dict().items()}
            params = [q for k, q in p.items() if "coord_mlp_vel" not in k]
            fwd = lambda: O.segno_forward(p, his, x, row, col, v, ea, T)[0]
        opt = torch.optim.Adam(params, lr=5e-3, weight_decay=1e-12)
        what = f"SEGNO N={N}, {T} sub-steps, dense-M segment mean included"

    def step():
        opt.zero_grad()
        loss = ((fwd() - target) ** 2).mean()
        loss.backward()
        opt.step()
        return float(loss.detach())

    sync = torch.cuda.synchronize if dev.type == "cuda" else (lambda: None)
    for _ in range(warmup):
        step()
    sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    sync()
    dt = time.perf_counter() - t0
    kind = "reference" if R is not None else "port"
    where = f"torch CPU fp32, {cores} threads" if dev.type == "cpu" else "torch eager fp32 on the B200 (TF32 off)"
    return {"value": sample * steps / dt, "unit": UNIT, "cores": cores if dev.type == "cpu" else 0, "kind": kind,
            "sample": f"{steps} steps x {sample} trajectories ({what}) fwd+bwd+Adam, {where}, {warmup} warm-up; "
                      + ("the reference's own nn.Module from oracle/_ref" if R is not None else "oracle port (oracle/nbody_oracle.py)"),
            "ms_per_step": 1e3 * dt / steps}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warmup = max(1, min(args.warmup, 2))
    cb = cpu_reference_arm(args, steps, warmup, args.cpu_sample)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, per_step=args.cpu_sample, note="CPU reference arm: bounded sample per step"),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def load_digest():
    """profiles/ncu_digest.json: per-kernel numbers read from committed ncu captures (tools/ncu_digest.py)."""
    path = os.path.join(ROOT, "profiles", "ncu_digest.json")
    try:
        with open(path) as fh:
            return json.load(fh)
    except Exception:
        return {}


def workload_config(args, per_step=None, note=None):
    c = {"workload": f"EGNO charged N-body, {args.n_balls} particles, num_timesteps={args.timesteps}, hidden 64, "
                     f"{args.layers} layers (BASELINE.json configs[2])",
         "batch_per_gpu": per_step if per_step is not None else args.batch, "n_balls": args.n_balls,
         "num_timesteps": args.timesteps, "n_layers": args.layers,
         "parallelism": f"dp{args.gpus}" + ("" if args.gpus == 1 else (" (NCCL all-reduce of the flat gradient bucket)" if os.environ.get("NB_BENCH_DP", "peer") == "nccl" else
                                                                       " (gradient sum over NVLink peer memory fused into the Adam kernel, no collective call)")), "launch": "eager" if args.no_graph else "cuda-graph replay (one graph per step)",
         "cache": "per-step activation working set (~270 MB at B=256) exceeds the 126 MB L2; inputs rotate over "
                  "8 distinct batches"}
    if note:
        c["note"] = note
    return c


# ------------------------------------------------------------------------------------------------ GPU arm
def finish(world, dist):
    """End of a rank: every rank reaches the barrier, then leaves without tearing NCCL down — destroying the process
    group while captured CUDA graphs still hold its collectives can block forever, and the process is exiting anyway."""
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def run_ours(args):
    import no_node_comparison_b200 as nb
    from no_node_comparison_b200 import synth
    from no_node_comparison_b200.dataparallel import init_from_env, broadcast_parameters
    import torch.distributed as dist
    import ctypes

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    rank, local, world = init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = nb.load_library()
    N, T, L, B = args.n_balls, args.timesteps, args.layers, args.batch
    K, W = args.steps, max(args.warmup, 3)

    torch.manual_seed(1)
    model = nb.EGNO(n_layers=L, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T,
                    device=dev)
    # data parallel: the gradient reduction is fused into the optimizer kernel over peer memory (NB_BENCH_DP=nccl selects
    # the NCCL flat-bucket all-reduce instead)
    peer_dp = os.environ.get("NB_BENCH_DP", "peer") != "nccl"
    if world > 1:
        broadcast_parameters(model)
        model.enable_data_parallel(peer_memory=peer_dp)
    use_graph = not args.no_graph
    opt = nb.FlatAdam(model.parameters(), lr=1e-4, weight_decay=1e-8, peer_bucket=model.peer_bucket)   # model_confs.yaml:15-17

    # ---- synthetic data: NB distinct batches per rank, raw states in pinned host memory
    NBATCH = 8
    row, col = synth.canonical_edges(B, N)
    row_d, col_d = row.to(dev), col.to(dev)
    edges = [row_d, col_d]
    t_out = torch.arange(1, T + 1, device=dev)[None].repeat(B, 1)
    host, resident = [], []
    F0 = 30      # input frame of the reference's loader for the charged data set (dataset_simple.py:123); targets = the next T
    for i in range(NBATCH):
        # synthetic trajectories of synthetic_sim.py's charged system, integrated by this repo's device simulator
        # (nb.simulate_charged, pinned to the reference by tests/test_sim.py) from its initial-condition distribution
        s0 = synth.sample_state("charged", B, N, seed=1000 * rank + i)
        f64 = lambda t: t.to(dev, torch.float64)
        loc_f, vel_f = nb.simulate_charged(f64(s0["loc"]).transpose(1, 2).contiguous(), f64(s0["vel"]).transpose(1, 2).contiguous(),
                                           f64(s0["charges"]), (F0 + T + 2) * 100, 100)        # [B, frames, 3, N]
        s = dict(loc=loc_f[:, F0].transpose(1, 2).float().cpu().contiguous(), vel=vel_f[:, F0].transpose(1, 2).float().cpu().contiguous(),
                 charges=s0["charges"])
        tgt = loc_f[:, F0 + 1:F0 + T + 1].permute(1, 0, 3, 2).reshape(T * B * N, 3).float().cpu()   # frame-major like the output
        hb = {k: v.contiguous().pin_memory() for k, v in dict(loc=s["loc"], vel=s["vel"], charges=s["charges"], target=tgt).items()}
        host.append(hb)
        x, nodes, ea, v, lm = synth.egno_features(s["loc"].to(dev), s["vel"].to(dev), s["charges"].to(dev), row_d, col_d)
        resident.append(dict(x=x, nodes=nodes, ea=ea, v=v, lm=lm, target=tgt.to(dev)))
    h2d_bytes = sum(t.numel() * t.element_size() for t in host[0].values())

    def loss_fn(x, nodes, ea, v, lm, target, keep=None):
        xo, vo, ho = model(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
        loss = nb.trajectory_mse(xo, target, T)[0]      # the callers' MSE (main_simulation_simple_no.py:273-276), fused
        if keep is not None:
            # --dump-outputs: detached views; under graph replay they are the graph's outputs, rewritten by every replay
            keep.update(loss=loss.detach(), x_out=xo.detach(), v_out=vo.detach(), h_out=ho.detach())
        return loss

    last = {}                   # the latest timed step's results (--dump-outputs)
    train_loss = functools.partial(loss_fn, keep=last) if args.dump_outputs else loss_fn

    def loss_from_raw(loc, vel, charges, target):
        # prepare_inputs on the device: one featurisation kernel (nb_nbody_features)
        x, v = loc.reshape(-1, 3), vel.reshape(-1, 3)
        nodes, lm, ea = nb.prepare_inputs(x, v, charges, N, with_charge=True)
        return loss_fn(x, nodes, ea, v, lm, target)

    def eager_step(b):
        opt.zero_grad(set_to_none=True)
        loss = train_loss(b["x"], b["nodes"], b["ea"], b["v"], b["lm"], b["target"])
        loss.backward()
        opt.step()
        return loss

    if use_graph:
        # one CUDA graph per step shape: forward + loss + backward (+ all-reduce) + Adam replayed as a single launch
        g_res = nb.GraphedStep(train_loss, {k: resident[0][k] for k in ("x", "nodes", "ea", "v", "lm", "target")}, opt)
        g_raw = nb.GraphedStep(loss_from_raw, {k: host[0][k].to(dev) for k in ("loc", "vel", "charges", "target")}, opt)

        def train_step(b):
            return g_res(**{k: b[k] for k in ("x", "nodes", "ea", "v", "lm", "target")})

        def e2e_step(hb):
            return g_raw(**hb).item()      # H2D from pinned memory into the graph's input buffers; D2H read of the loss
    else:
        train_step = eager_step

        def e2e_step(hb):
            d = {k: t.to(dev, non_blocking=True) for k, t in hb.items()}              # H2D from pinned memory
            loss = loss_from_raw(d["loc"], d["vel"], d["charges"], d["target"])
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            return loss.item()                                                         # D2H read of the step's loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(W):
        train_step(resident[i % NBATCH])
    l0 = lib.nb_launch_count()
    tw0 = time.time()
    ms = timed(lambda i: train_step(resident[i % NBATCH]), K)
    tw1 = time.time()
    launches = lib.nb_launch_count() - l0
    if use_graph:   # replays do not pass through the library's host-side counter: kernels per captured step x K
        launches = g_res.launches_per_replay * K
    clocks = sampler.stop(window=(tw0, tw1)) if rank == 0 else None
    value = world * B * K / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        ps = list(model.parameters())                 # the optimizer's parameter order
        gs = g_res.grads if use_graph else [p.grad for p in ps]
        last["params"] = torch.cat([p.detach().reshape(-1) for p in ps])
        last["grads"] = torch.cat([(torch.zeros_like(p) if g is None else g.detach()).reshape(-1) for p, g in zip(ps, gs)])
        dump_outputs(args.dump_outputs, last)

    if args.quick:
        lib.nb_profile_enable(1)
        ms_q = timed(lambda i: eager_step(resident[i % NBATCH]), K)
        qm, qc = (ctypes.c_double * 8)(), (ctypes.c_longlong * 8)()
        lib.nb_profile_read(qm, qc)
        lib.nb_profile_enable(0)
        per = {c: round(1e3 * qm[i] / max(qc[i], 1), 1)
               for c, i in {"edge_fwd": 0, "edge_bwd": 1, "node": 2, "wgrad64": 3, "tconv": 4, "node_fwd": 6, "node_bwd": 7}.items()}
        if rank == 0:
            emit(dict({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                              "ms_per_step": ms / K, "gpu_launches": int(launches), "quick": True,
                              "us_per_launch": per, "ms_in_kernels_per_step": round(sum(qm[:5]) / K, 3)}))
        finish(world, dist)
        return

    # ---- end to end: host buffers in, loss out, through the module API
    for i in range(2):
        e2e_step(host[i % NBATCH])
    ms_e2e = timed(lambda i: e2e_step(host[i % NBATCH]), K)
    e2e_value = world * B * K / (ms_e2e / 1e3)

    # ---- per-kernel CUDA-event timing (separate pass so the events do not perturb `value`)
    # (eager launches: the per-kernel events are recorded by the library's host-side launch code, which a graph replay skips)
    lib.nb_profile_enable(1)
    ms_prof = timed(lambda i: eager_step(resident[i % NBATCH]), K)
    pm = (ctypes.c_double * 8)()
    pc = (ctypes.c_longlong * 8)()
    lib.nb_profile_read(pm, pc)
    lib.nb_profile_enable(0)
    cats = {"edge_fwd": 0, "edge_bwd": 1, "node": 2, "wgrad64": 3, "tconv": 4, "node_fwd": 6, "node_bwd": 7}
    kern = {c: {"ms_total": pm[i], "launches": int(pc[i]), "ms_per_launch": (pm[i] / pc[i]) if pc[i] else None,
                "share_of_step": pm[i] / ms_prof if ms_prof else None} for c, i in cats.items()}

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        pk = json.load(open(peaks_path))
        peak_tf, peak_src = float(pk["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        hbm = float(pk["hbm_gbs"])
    else:
        peak_tf, peak_src, hbm = 1400.0, "fallback (B200_PROFILING.md sustained bf16)", 6650.0
    ne = T * B * N * (N - 1)
    digest = load_digest()
    dg = digest.get("k_edge_bwd_sel", {}) if (N, T, B) == (20, 10, 256) else {}
    t_bwd = kern["edge_bwd"]["ms_per_launch"]
    flop_kernel = 2 * 2 * MAC_EDGE_KERNEL * ne           # backward = 2 x forward; recompute is not credited
    achieved = flop_kernel / (t_bwd * 1e-3) / 1e12 if t_bwd else None
    roofline = {"kernel": "k_edge_bwd_sel (fused E_GCL edge-tile backward: recompute + dgrad + wgrad + node gathers/scatters, "
                          "all on tcgen05 with split-bf16 operands and fp32 TMEM accumulators)",
                "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": (achieved / peak_tf) if achieved else None, "peak_source": peak_src,
                # every logical fp32 product is three bf16 passes: the ceiling for fp32-accurate work on this pipe
                "peak_3pass": peak_tf / 3.0, "frac_3pass": (achieved / (peak_tf / 3.0)) if achieved else None,
                "frac_reference_formula": (2 * 2 * MAC_EDGE_REF * ne / (t_bwd * 1e-3) / 1e12 / peak_tf) if t_bwd else None,
                # dram__bytes_read.sum + dram__bytes_write.sum per launch and tensor-pipe activity from the committed ncu
                # digest of this kernel (profiles/ncu_digest.json, written by tools/ncu_digest.py); default workload only
                "traffic": dg.get("dram_bytes"), "tensor_pipe_active_pct_ncu": dg.get("tensor_pipe_active_pct"),
                "ncu_source": dg.get("source"),
                "flop_per_launch": flop_kernel, "flop_per_launch_reference_formula": 2 * 2 * MAC_EDGE_REF * ne,
                "note": "achieved = ALGORITHMIC fp32 FLOPs the edge kernel owns (8448 MAC/edge forward, x2 for backward; the "
                        "recompute is not credited) / its mean launch time (CUDA events on the launch stream).  The reference's "
                        "dense 131-wide first layer would count 16640 MAC/edge (second figure).  Every logical fp32 MMA is "
                        "three bf16 tcgen05 passes (hi*hi + lo*hi + hi*lo) and the backward executes ~2x the credited MACs "
                        "(recompute, weight-gradient and one-hot scatter MMAs), so the tensor pipe is ~8x busier than `frac` "
                        "suggests (tensor_pipe_active_pct_ncu).  frac_3pass is the same figure against peak / 3, the ceiling "
                        "of fp32-accurate products on this pipe.  Not HBM-bound: `traffic` is ~1.1x the node-level bytes.",
                "hbm_peak_gbs": hbm}

    # HBM-bound side of the path: the fused temporal convolution (forward reads h and writes h once; the backward reads h
    # and dL/dh_out, writes dL/dh_in and the 2 x 3 coefficient planes the weight-gradient reduction consumes)
    nn0 = B * N
    tconv_bytes_fwd = 2 * T * nn0 * 64 * 4
    tconv_bytes_bwd = 3 * T * nn0 * 64 * 4 + 2 * 3 * nn0 * 64 * 4
    t_tc = kern["tconv"]["ms_per_launch"]
    tc_ach = 0.5 * (tconv_bytes_fwd + tconv_bytes_bwd) / (t_tc * 1e-3) / 1e9 if t_tc else None
    roofline_hbm = {"kernel": "k_tconv_fwd / k_tconv_bwd (fused DFT + fp32 mode mixing + inverse DFT + LeakyReLU/residual)",
                    "bound": "hbm", "achieved": tc_ach, "peak": hbm, "unit": "GB/s", "frac": (tc_ach / hbm) if tc_ach else None,
                    "bytes_per_launch_fwd": tconv_bytes_fwd, "bytes_per_launch_bwd": tconv_bytes_bwd,
                    "note": "mean over the forward and backward launches of a step (CUDA events); algorithmic bytes = "
                            "2*T*64*4 B per node-trajectory forward, (3*T + 6)*64*4 B backward"}

    # the per-layer node kernels (nb_egno_node.cuh): every tensor crosses HBM once per kernel
    rows = T * nn0
    nf_bytes = rows * 4 * (2 * 64 + 3 * 3 + 3 * 64 + 3)           # reads h, M, x, v, Fsum ; writes U5, UV, h', x'
    nb_bytes = rows * 4 * (3 * 64 + 4 * 3 + 4 * 64 + 2 * 3)       # reads gh, U5, UV, gx, gv, v, Fsum ; writes GUV, GU5, gh1, gM, gv, gFsum
    t_nf, t_nb = kern["node_fwd"]["ms_per_launch"], kern["node_bwd"]["ms_per_launch"]
    roofline_node = None
    if t_nf and t_nb:
        roofline_node = {"kernel": "k_egno_node_fwd / k_egno_node_bwd (node_net + node_v_net + coordinate update of a layer, "
                                   "operands chained through tensor memory)",
                         "bound": "hbm", "peak": hbm, "unit": "GB/s",
                         "achieved_fwd": nf_bytes / (t_nf * 1e-3) / 1e9, "achieved_bwd": nb_bytes / (t_nb * 1e-3) / 1e9,
                         "frac_fwd": nf_bytes / (t_nf * 1e-3) / 1e9 / hbm, "frac_bwd": nb_bytes / (t_nb * 1e-3) / 1e9 / hbm,
                         "bytes_per_launch_fwd": nf_bytes, "bytes_per_launch_bwd": nb_bytes,
                         "traffic_fwd": (digest.get("k_egno_node_fwd") or {}).get("dram_bytes"),
                         "traffic_bwd": (digest.get("k_egno_node_bwd") or {}).get("dram_bytes"),
                         "ncu_source": (digest.get("k_egno_node_fwd") or {}).get("source"),
                         "note": "algorithmic bytes = the kernel's inputs and outputs once (rows = T*B*N); live CUDA-event time per launch"}

    extras, segno = {}, None
    if not args.no_extras:
        # inference throughput (no_grad forward) of the same model
        with torch.no_grad():
            f = lambda i: model(resident[i % NBATCH]["x"], resident[i % NBATCH]["nodes"], edges, resident[i % NBATCH]["ea"],
                                v=resident[i % NBATCH]["v"], loc_mean=resident[i % NBATCH]["lm"], timesteps_out=t_out)
            for i in range(3):
                f(i)
            ms_inf = timed(f, K)
        extras["egno_infer_traj_per_s"] = world * B * K / (ms_inf / 1e3)
        # SEGNO, BASELINE.json configs[3] shape (gravity, N=20, 10 sub-steps, B=256): the second half of the metric
        torch.manual_seed(1)
        seg = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=dev, n_layers=8, recurrent=True)
        if world > 1:
            broadcast_parameters(seg)
            seg.enable_data_parallel(peer_memory=peer_dp)
        sopt = nb.FlatAdam(seg.parameters(), lr=5e-3, weight_decay=1e-12, peer_bucket=seg.peer_bucket)
        sb, shost = [], []
        for i in range(NBATCH):
            # trajectories of synthetic_sim.py's gravitational system (nb.simulate_gravity): frame 0 in, frame 1 out
            s0 = synth.sample_state("gravity", B, N, seed=77 + 1000 * rank + i)
            f64 = lambda t: t.to(dev, torch.float64)
            pos_f, vel_f, _ = nb.simulate_gravity(f64(s0["loc"]), f64(s0["vel"]), f64(s0["charges"]), 200, 100)   # [B, 2, N, 3]
            loc0, vel0 = pos_f[:, 0].float().contiguous(), vel_f[:, 0].float().contiguous()
            tgt = pos_f[:, 1].float().reshape(B * N, 3).contiguous()
            his, x, v, ea = synth.segno_features(loc0, vel0, s0["charges"].to(dev), row_d, col_d)
            sb.append(dict(his=his, x=x, v=v, ea=ea, target=tgt))
            shost.append({k: t.cpu().contiguous().pin_memory() for k, t in dict(loc=loc0, vel=vel0, mass=s0["charges"], target=tgt).items()})
        seg_h2d = sum(t.numel() * t.element_size() for t in shost[0].values())

        def seg_loss(his, x, v, ea, target):
            xo, ho, vo = seg(his, x, edges, v, ea, T=T)
            return nb.trajectory_mse(xo, target, 1)[0]          # MSELoss()(loc_pred, loc_end), train_nbody.py:163-165, fused

        def seg_loss_raw(loc, vel, mass, target):
            x, v = loc.reshape(-1, 3), vel.reshape(-1, 3)
            his, _, ea = nb.prepare_inputs(x, v, mass, N, with_charge=False, want_mean=False)    # train_nbody.py:93,119-123
            return seg_loss(his, x, v, ea, target)

        def seg_eager(i):
            sopt.zero_grad(set_to_none=True)
            seg_loss(**sb[i % NBATCH]).backward()
            sopt.step()

        if use_graph:
            g_seg = nb.GraphedStep(seg_loss, sb[0], sopt)
            g_seg_raw = nb.GraphedStep(seg_loss_raw, {k: t.to(dev) for k, t in shost[0].items()}, sopt)
            seg_step = lambda i: g_seg(**sb[i % NBATCH])
            seg_e2e = lambda i: g_seg_raw(**shost[i % NBATCH]).item()
            seg_launches = g_seg.launches_per_replay
        else:
            seg_step = seg_eager

            def seg_e2e(i):
                d = {k: t.to(dev, non_blocking=True) for k, t in shost[i % NBATCH].items()}
                sopt.zero_grad(set_to_none=True)
                loss = seg_loss_raw(**d)
                loss.backward()
                sopt.step()
                return loss.item()
            seg_launches = None

        for i in range(3):
            seg_step(i)
        ms_seg = timed(seg_step, K)
        for i in range(2):
            seg_e2e(i)
        ms_seg_e2e = timed(seg_e2e, K)
        with torch.no_grad():
            g = lambda i: seg(sb[i % NBATCH]["his"], sb[i % NBATCH]["x"], edges, sb[i % NBATCH]["v"], sb[i % NBATCH]["ea"], T=T)
            for i in range(3):
                g(i)
            ms_sinf = timed(g, K)
        lib.nb_profile_enable(1)
        ms_sprof = timed(seg_eager, K)
        sm_, sc_ = (ctypes.c_double * 8)(), (ctypes.c_longlong * 8)()
        lib.nb_profile_read(sm_, sc_)
        lib.nb_profile_enable(0)
        scat = {"edge_bwd": 1, "segno_fused_fwd": 5, "node": 2, "wgrad64": 3}
        skern = {c: {"ms_total": sm_[i], "launches": int(sc_[i]), "ms_per_launch": (sm_[i] / sc_[i]) if sc_[i] else None,
                     "share_of_step": sm_[i] / ms_sprof if ms_sprof else None} for c, i in scat.items()}
        ne_s = B * N * (N - 1)                                    # edges per sub-step
        t_sb, t_sf = skern["edge_bwd"]["ms_per_launch"], skern["segno_fused_fwd"]["ms_per_launch"]
        mac_node = 2 * 64 * 64 + 2 * 64 * 64 + 64 * 64            # P|Q, phi_h first layer ([h, M] 128-wide), second layer
        flop_fused = 2 * T * (MAC_EDGE_KERNEL * ne_s + mac_node * B * N)
        flop_sbwd = 2 * 2 * MAC_EDGE_KERNEL * ne_s
        tf = lambda fl, ms_: fl / (ms_ * 1e-3) / 1e12 if ms_ else None
        segno = {"config": {"workload": f"SEGNO gravity N-body, {N} particles, {T} sub-steps, hidden 64 (BASELINE.json configs[3])",
                            "batch_per_gpu": B},
                 "train_traj_per_s": world * B * K / (ms_seg / 1e3), "ms_per_step": ms_seg / K,
                 "infer_traj_per_s": world * B * K / (ms_sinf / 1e3),
                 "e2e": {"value": world * B * K / (ms_seg_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": seg_h2d,
                         "d2h_bytes_per_step": 4, "ms_per_step": ms_seg_e2e / K},
                 "gpu_launches_per_step": seg_launches,
                 "roofline": {"kernel": "k_edge_bwd_sel at the SEGNO shape (one launch per sub-step of the backward sweep; "
                                        f"{ne_s} edges = {-(-ne_s // 128)} tiles over the SMs)",
                              "bound": "tensor", "achieved": tf(flop_sbwd, t_sb), "peak": peak_tf, "unit": "TFLOP/s",
                              "frac": (tf(flop_sbwd, t_sb) / peak_tf) if t_sb else None,
                              "frac_3pass": (tf(flop_sbwd, t_sb) / (peak_tf / 3)) if t_sb else None, "peak_source": peak_src,
                              "traffic": digest.get("k_edge_bwd_sel_segno", {}).get("dram_bytes"),
                              "ncu_source": digest.get("k_edge_bwd_sel_segno", {}).get("source")},
                 "roofline_fused_fwd": {"kernel": "k_segno_fused_fwd (all sub-steps of the forward in one kernel, node state in "
                                                  "shared memory)", "bound": "tensor", "achieved": tf(flop_fused, t_sf),
                                        "peak": peak_tf, "unit": "TFLOP/s", "frac": (tf(flop_fused, t_sf) / peak_tf) if t_sf else None,
                                        "frac_3pass": (tf(flop_fused, t_sf) / (peak_tf / 3)) if t_sf else None,
                                        "traffic": digest.get("k_segno_fused_fwd", {}).get("dram_bytes"),
                                        "tensor_pipe_active_pct_ncu": digest.get("k_segno_fused_fwd", {}).get("tensor_pipe_active_pct"),
                                        "ncu_source": digest.get("k_segno_fused_fwd", {}).get("source"),
                                        "note": f"one CTA per trajectory: {B} CTAs on {torch.cuda.get_device_properties(dev).multi_processor_count} SMs"},
                 "kernels": skern}
        extras["segno_train_traj_per_s"] = segno["train_traj_per_s"]
        extras["segno_infer_traj_per_s"] = segno["infer_traj_per_s"]
        # long-horizon rollouts kept on the device (featurisation + model + energies; BASELINE.json configs[3]:
        # traj_len = 20 calls, main.py:42), one host read at the end
        TL = 20
        s0 = synth.sample_state("gravity", B, N, seed=4242 + rank)
        l0_, v0_, m0_ = (s0[k].reshape(B * N, -1).to(dev) for k in ("loc", "vel", "charges"))
        ro = lambda i: nb.segno_rollout(seg, l0_, v0_, m0_, edges, N, traj_len=TL, num_steps=T, dataset="gravity")[1].sum().item()
        ro(0)
        ms_ro = timed(ro, 3)
        extras["segno_rollout_traj_per_s"] = world * B * 3 / (ms_ro / 1e3)
        extras["segno_rollout_note"] = f"{TL} autoregressive calls x {T} sub-steps + energy of every frame per trajectory"
        c0 = synth.sample_state("charged", B, N, seed=777 + rank)
        cl, cv, cq = (c0[k].reshape(B * N, -1).to(dev) for k in ("loc", "vel", "charges"))
        er = lambda i: nb.egno_rollout(model, cl, cv, cq, edges, N, traj_len=TL, dataset="charged")[2].sum().item()
        er(0)
        ms_er = timed(er, 3)
        extras["egno_rollout_traj_per_s"] = world * B * 3 / (ms_er / 1e3)
        extras["egno_rollout_note"] = f"{TL} autoregressive calls x {T} frames + energy of every frame per trajectory"
        # the two 5-body configurations (BASELINE.json configs[0], configs[1]): launch-bound, so one CUDA graph per step
        if world == 1:
            extras.update(small_configs(nb, synth, dev, K))

    # ---- BASELINE.json configs[4]: 100-body EGNO, GLOBAL batch 512 split over the ranks (strong scaling), at every N
    cfg5 = None
    if not args.no_extras:
        cfg5 = config5_leg(nb, synth, dev, rank, world, timed, dist, use_graph)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_arm(args, steps=8, warmup=1, sample=args.cpu_sample)
        cpu_baseline = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if not args.no_extras:
            # same-GPU context (SURVEY.md 0): the plain PyTorch eager ops of the oracle port on this B200, same config
            try:
                eg = cpu_reference_arm(args, steps=5, warmup=2, sample=B, device="cuda")
                cpu_baseline["torch_eager_b200"] = {"value": eg["value"], "unit": UNIT, "sample": eg["sample"]}
                extras["torch_eager_b200_traj_per_s"] = eg["value"]
            except Exception as e:
                cpu_baseline["torch_eager_b200"] = {"error": str(e)[:200]}
            cs = cpu_reference_arm(args, steps=8, warmup=1, sample=args.cpu_sample, model="segno")
            segno["cpu_baseline"] = {k: cs[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic (trajectories of the reference's charged simulator, integrated on the device)",
                "config": workload_config(args), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / K},
                "gpu_launches": int(launches), "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_node": roofline_node,
                "cpu_baseline": cpu_baseline,
                "kernels": kern,
                "kernels_note": "CUDA-event time per launch category of an eager pass; wgrad64 (and the finalisations) run on "
                                "the library's second stream underneath the next layer's kernels, so its launch time is "
                                "stretched by the overlap, node_bwd shares the SMs with it, and the shares need not add up to 1",
                "segno": segno, "config5": cfg5, "extras": extras}
        emit(line)
    finish(world, dist)


def config5_leg(nb, synth, dev, rank, world, timed, dist, use_graph):
    """BASELINE.json configs[4]: EGNO on a synthetic 100-particle charged system, batch 512, data-parallel over the ranks
    (strong scaling: 512 / world trajectories per GPU; one flat-bucket all-reduce per step)."""
    GB, N5, T5, L5 = 512, 100, 10, 4
    B5 = GB // world
    row5, col5 = synth.canonical_edges(B5, N5)
    e5 = [row5.to(dev), col5.to(dev)]
    torch.manual_seed(1)
    m5 = nb.EGNO(n_layers=L5, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T5, device=dev)
    if world > 1:
        from no_node_comparison_b200.dataparallel import broadcast_parameters

        broadcast_parameters(m5)
        m5.enable_data_parallel(peer_memory=os.environ.get("NB_BENCH_DP", "peer") != "nccl")
    o5 = nb.FlatAdam(m5.parameters(), lr=1e-4, weight_decay=1e-8, peer_bucket=m5.peer_bucket)
    s5 = synth.sample_state("charged", B5, N5, seed=9 + rank)
    x5, n5, ea5, v5, lm5 = synth.egno_features(s5["loc"].to(dev), s5["vel"].to(dev), s5["charges"].to(dev), e5[0], e5[1])
    tg5 = x5.repeat(T5, 1) + 0.05 * torch.randn(T5 * B5 * N5, 3, device=dev)
    to5 = torch.arange(1, T5 + 1, device=dev)[None].repeat(B5, 1)

    def loss5(x, nodes, ea, v, lm, tgt):
        xo, _, _ = m5(x, nodes, e5, ea, v=v, loc_mean=lm, timesteps_out=to5)
        return nb.trajectory_mse(xo, tgt, T5)[0]

    ins = dict(x=x5, nodes=n5, ea=ea5, v=v5, lm=lm5, tgt=tg5)
    if use_graph:
        g5 = nb.GraphedStep(loss5, ins, o5, warmup=2)
        step5 = lambda i: g5.graph.replay()
    else:
        def step5(i):
            o5.zero_grad(set_to_none=True)
            loss5(**ins).backward()
            o5.step()
        for _ in range(2):
            step5(0)
    K5 = 5
    ms5 = timed(step5, K5)
    out = {"workload": "EGNO synthetic 100-particle charged system, batch 512, data-parallel (BASELINE.json configs[4])",
           "metric": "train trajectories/s (EGNO 100-body, fwd+bwd+Adam)", "value": GB * K5 / (ms5 / 1e3), "unit": UNIT,
           "scaling": "strong", "global_batch": GB, "batch_per_gpu": B5, "n_gpus": world, "steps": K5,
           "ms_per_step": ms5 / K5, "edges_per_layer_per_gpu": T5 * B5 * N5 * (N5 - 1),
           "data": "synthetic (initial-condition distribution of the charged simulator; runtime is value-independent)"}
    del m5, o5
    torch.cuda.empty_cache()
    return out


def small_configs(nb, synth, dev, K):
    """Training throughput of the 5-body configurations: EGNO N=5, T=8, L=4, B=100 and SEGNO N=5, T=10, B=100."""
    out = {}
    B, N = 100, 5
    row, col = synth.canonical_edges(B, N)
    edges = [row.to(dev), col.to(dev)]

    def run(step, n):
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            step()
        e1.record()
        torch.cuda.synchronize()
        return B * n / (e0.elapsed_time(e1) / 1e3)

    T = 8
    torch.manual_seed(1)
    m = nb.EGNO(n_layers=4, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T, device=dev)
    opt = nb.FlatAdam(m.parameters(), lr=1e-4, weight_decay=1e-8)
    s = synth.sample_state("charged", B, N, seed=5)
    x, nodes, ea, v, lm = synth.egno_features(s["loc"].to(dev), s["vel"].to(dev), s["charges"].to(dev), edges[0], edges[1])
    tgt = x.repeat(T, 1) + 0.05 * torch.randn(T * B * N, 3, device=dev)
    t_out = torch.arange(1, T + 1, device=dev)[None].repeat(B, 1)

    def f1(x, nodes, ea, v, lm, tgt):
        xo, _, _ = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
        return ((xo - tgt) ** 2).mean()

    ins = dict(x=x, nodes=nodes, ea=ea, v=v, lm=lm, tgt=tgt)
    g1 = nb.GraphedStep(f1, ins, opt)
    out["egno_n5_t8_b100_train_traj_per_s"] = run(lambda: g1(**ins), 4 * K)
    T2 = 10
    torch.manual_seed(1)
    sg = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=dev, n_layers=8, recurrent=True)
    sopt = nb.FlatAdam(sg.parameters(), lr=5e-3, weight_decay=1e-12)
    his, x2, v2, ea2 = synth.segno_features(s["loc"].to(dev), s["vel"].to(dev), s["charges"].to(dev), edges[0], edges[1])
    tgt2 = x2 + 0.05 * torch.randn_like(x2)

    def f2(his, x, v, ea, tgt):
        xo, _, _ = sg(his, x, edges, v, ea, T=T2)
        return ((xo - tgt) ** 2).mean()

    ins2 = dict(his=his, x=x2, v=v2, ea=ea2, tgt=tgt2)
    g2 = nb.GraphedStep(f2, ins2, sopt)
    out["segno_n5_t10_b100_train_traj_per_s"] = run(lambda: g2(**ins2), 4 * K)
    out["small_configs_note"] = "BASELINE.json configs[0] / [1] (B=100): launch-bound; whole step replayed as one CUDA graph"
    del g1, g2, m, sg
    return out


def main():
    args = parse()
    # stdout carries exactly ONE JSON line: libraries that print to file descriptor 1 (NCCL's "NCCL version ..." banner when
    # NCCL_DEBUG is set in the environment) are sent to stderr; emit() writes the line to the real stdout
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
