"""Generate golden vectors from the REAL reference (needs it installed: oracle/make_ref.py).

    python tests/golden/make_golden.py

Imports the reference through oracle/ref_loader.py (stubs for torch_geometric /
matplotlib only), simulates a few trajectories with the reference's own
``synthetic_sim`` (np.random.seed(43), README.md:6), builds features the way the
reference callers do, runs the reference ``EGNO`` module and ``SEGNO.forward_step``
with ``torch.manual_seed(1)`` weights, and stores inputs, weights, outputs and
gradients as ``tests/golden/<case>.npz``.  The gradients are those of
``L = <x_out,Gx> + <v_out,Gv> + <h_out,Gh>`` for seeded cotangents G* (stored).

The reference has no tests or fixtures of its own (SURVEY.md §4), so these files
are the pin for both the oracle restatement and the CUDA path.
"""
from __future__ import annotations

import io
import contextlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from oracle import nbody_oracle as O  # noqa: E402


def simulate(ref, kind: str, n_balls: int, n_traj: int, length: int = 5000, sample_freq: int = 100):
    """-> loc, vel [S, frames, N, 3] float32 ; charges/masses [S, N, 1]."""
    ss = ref.synthetic_sim
    with contextlib.redirect_stdout(io.StringIO()):
        if kind == "charged":
            sim = ss.ChargedParticlesSim(noise_var=0.0, n_balls=n_balls, vel_norm=0.5)
        else:
            sim = ss.GravitySim(noise_var=0.0, n_balls=n_balls, vel_norm=0.5)
    locs, vels, qs = [], [], []
    for _ in range(n_traj):
        loc, vel, _, q = sim.sample_trajectory(T=length, sample_freq=sample_freq)
        if kind == "charged":           # [frames, 3, N] -> [frames, N, 3]  (dataset_simple.py:43-47)
            loc, vel = loc.transpose(0, 2, 1), vel.transpose(0, 2, 1)
        locs.append(loc), vels.append(vel), qs.append(q)
    return (np.stack(locs).astype(np.float32), np.stack(vels).astype(np.float32),
            np.stack(qs).astype(np.float32))


def cot(shape, gen):
    return torch.randn(shape, generator=gen)


def run_egno(ref, name, n_balls, B, T, n_layers, num_modes, frame0=30):
    np.random.seed(43)
    loc, vel, q = simulate(ref, "charged", n_balls, B)
    loc0, vel0 = torch.tensor(loc[:, frame0]), torch.tensor(vel[:, frame0])
    row, col = O.canonical_edges(B, n_balls)
    x, v, edge_attr, nodes, loc_mean = O.egno_features(loc0, vel0, torch.tensor(q), row, col)
    torch.manual_seed(1)
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref.EGNO(n_layers=n_layers, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, flat=False,
                         norm=False, num_modes=num_modes, num_timesteps=T, time_emb_dim=32, num_inputs=1,
                         device="cpu")
    t_out = torch.arange(1, T + 1)[None].repeat(B, 1)
    x = x.clone().requires_grad_(True)
    v = v.clone().requires_grad_(True)
    xo, vo, ho = model(x, nodes, [row, col], edge_attr, v=v, loc_mean=loc_mean, timesteps_out=t_out)
    gen = torch.Generator().manual_seed(7)
    Gx, Gv, Gh = cot(xo.shape, gen), cot(vo.shape, gen), cot(ho.shape, gen) * 0.1
    ((xo * Gx).sum() + (vo * Gv).sum() + (ho * Gh).sum()).backward()
    out = dict(meta=np.array([n_balls, B, T, n_layers, num_modes], dtype=np.int64),
               loc=loc0.numpy(), vel=vel0.numpy(), charges=q, t_out=t_out.numpy(),
               x_out=xo.detach().numpy(), v_out=vo.detach().numpy(), h_out=ho.detach().numpy(),
               Gx=Gx.numpy(), Gv=Gv.numpy(), Gh=Gh.numpy(),
               gx_in=x.grad.numpy(), gv_in=v.grad.numpy())
    for k, p in model.state_dict().items():
        out["w:" + k] = p.numpy()
    for k, p in model.named_parameters():
        out["g:" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "x_out", tuple(xo.shape), "params", sum(p.numel() for p in model.parameters()))


def run_egno_multi(ref, name, n_balls, B, T, n_layers, num_modes, num_inputs, var_dt, frames):
    """num_inputs > 1 (the PRO sweep, _schedule.yaml:38-68): several input frames, optional per-trajectory output times."""
    np.random.seed(43)
    loc, vel, q = simulate(ref, "charged", n_balls, B)
    locL = torch.tensor(loc[:, frames]).transpose(0, 1).contiguous()   # [L,B,N,3]
    velL = torch.tensor(vel[:, frames]).transpose(0, 1).contiguous()
    row, col = O.canonical_edges(B, n_balls)
    x, v, edge_attr, nodes, loc_mean = O.egno_features_multi(locL, velL, torch.tensor(q), row, col)
    torch.manual_seed(1)
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref.EGNO(n_layers=n_layers, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, flat=False,
                         norm=False, num_modes=num_modes, num_timesteps=T, time_emb_dim=32, num_inputs=num_inputs,
                         varDT=var_dt, device="cpu")
    gen = torch.Generator().manual_seed(11)
    t_in = torch.arange(-num_inputs + 1, 1)[None].repeat(B, 1)
    if var_dt:   # per-trajectory ascending output times (utils.py:15-31 random_ascending_tensor)
        t_out = torch.stack([torch.sort(torch.randperm(3 * T, generator=gen)[:T] + 1).values for _ in range(B)])
    else:
        t_out = torch.arange(1, T + 1)[None].repeat(B, 1)
    x = x.clone().requires_grad_(True)
    v = v.clone().requires_grad_(True)
    xo, vo, ho = model(x, nodes, [row, col], edge_attr, v=v, loc_mean=loc_mean, timesteps_in=t_in, timesteps_out=t_out)
    gen = torch.Generator().manual_seed(7)
    Gx, Gv, Gh = cot(xo.shape, gen), cot(vo.shape, gen), cot(ho.shape, gen) * 0.1
    ((xo * Gx).sum() + (vo * Gv).sum() + (ho * Gh).sum()).backward()
    out = dict(meta=np.array([n_balls, B, T, n_layers, num_modes, num_inputs], dtype=np.int64),
               loc=locL.numpy(), vel=velL.numpy(), charges=q, t_out=t_out.numpy(), t_in=t_in.numpy(),
               x_out=xo.detach().numpy(), v_out=vo.detach().numpy(), h_out=ho.detach().numpy(),
               Gx=Gx.numpy(), Gv=Gv.numpy(), Gh=Gh.numpy(),
               gx_in=x.grad.numpy(), gv_in=v.grad.numpy())
    for k, p in model.state_dict().items():
        out["w:" + k] = p.numpy()
    for k, p in model.named_parameters():
        out["g:" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "x_out", tuple(xo.shape), "params", sum(p.numel() for p in model.parameters()))


def run_segno(ref, name, kind, n_balls, B, T, frame0):
    np.random.seed(43)
    loc, vel, q = simulate(ref, kind, n_balls, B)
    loc0, vel0 = torch.tensor(loc[:, frame0]), torch.tensor(vel[:, frame0])
    row, col = O.canonical_edges(B, n_balls)
    his, x, v, edge_attr = O.segno_features(loc0, vel0, torch.tensor(q), row, col)
    torch.manual_seed(1)
    model = ref.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", n_layers=8, recurrent=True,
                      norm_diff=False, tanh=False)
    x = x.clone().requires_grad_(True)
    v = v.clone().requires_grad_(True)
    # the intended semantics: forward_step(embedding(his)) -- SEGNO/models/model.py:73,95-102
    xo, ho, vo = model.forward_step(model.embedding(his), x, [row, col], v, edge_attr, T=T)
    gen = torch.Generator().manual_seed(7)
    Gx, Gv, Gh = cot(xo.shape, gen), cot(vo.shape, gen), cot(ho.shape, gen) * 0.1
    ((xo * Gx).sum() + (vo * Gv).sum() + (ho * Gh).sum()).backward()
    out = dict(meta=np.array([n_balls, B, T], dtype=np.int64), loc=loc0.numpy(), vel=vel0.numpy(), charges=q,
               x_out=xo.detach().numpy(), v_out=vo.detach().numpy(), h_out=ho.detach().numpy(),
               Gx=Gx.numpy(), Gv=Gv.numpy(), Gh=Gh.numpy(), gx_in=x.grad.numpy(), gv_in=v.grad.numpy())
    for k, p in model.state_dict().items():
        out["w:" + k] = p.numpy()
    for k, p in model.named_parameters():
        out["g:" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "x_out", tuple(xo.shape), "params", sum(p.numel() for p in model.parameters()))


def run_segno_multi(ref, name, n_balls, B, T, frames, agg):
    """Several input frames (model.py:65-90).  HEAD's forward returns the last segment's inputs (SURVEY.md 0); the
    vectors pin the intended result, computed with the reference's own forward_step / prepare_node_inputs."""
    np.random.seed(43)
    loc, vel, q = simulate(ref, "charged", n_balls, B)
    locL = torch.tensor(loc[:, frames]).transpose(0, 1).contiguous()
    velL = torch.tensor(vel[:, frames]).transpose(0, 1).contiguous()
    row, col = O.canonical_edges(B, n_balls)
    his, x, v, edge_attr = O.segno_features_multi(locL, velL, torch.tensor(q), row, col)
    torch.manual_seed(1)
    model = ref.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", n_layers=8, recurrent=True,
                      norm_diff=False, tanh=False, multiple_agg=agg)
    in_steps = torch.tensor([f - frames[0] for f in frames])
    x = x.clone().requires_grad_(True)
    v = v.clone().requires_grad_(True)
    steps = torch.diff(in_steps).tolist() + [T]
    h = model.embedding(his)
    h_, x_, v_ = h[:, 0, :], x[:, 0, :], v[:, 0, :]
    for i, step in enumerate(steps):
        xi, hi, vi = model.forward_step(h_, x_, [row, col], v_, edge_attr, T=step)
        if i < len(steps) - 1:
            if agg == "sum":
                h_, x_, v_ = h[:, i + 1, :] + hi, x[:, i + 1, :] + xi, v[:, i + 1, :] + vi
            else:
                x_, v_, h_ = model.prepare_node_inputs(torch.stack([x[:, i + 1, :], xi], dim=1),
                                                       torch.stack([v[:, i + 1, :], vi], dim=1),
                                                       torch.stack([h[:, i + 1, :], hi], dim=1))
    xo, ho, vo = xi, hi, vi
    gen = torch.Generator().manual_seed(7)
    Gx, Gv, Gh = cot(xo.shape, gen), cot(vo.shape, gen), cot(ho.shape, gen) * 0.1
    ((xo * Gx).sum() + (vo * Gv).sum() + (ho * Gh).sum()).backward()
    out = dict(meta=np.array([n_balls, B, T, len(frames)], dtype=np.int64), loc=locL.numpy(), vel=velL.numpy(), charges=q,
               in_steps=in_steps.numpy(), agg=np.array([0 if agg == "sum" else 1]),
               x_out=xo.detach().numpy(), v_out=vo.detach().numpy(), h_out=ho.detach().numpy(),
               Gx=Gx.numpy(), Gv=Gv.numpy(), Gh=Gh.numpy(), gx_in=x.grad.numpy(), gv_in=v.grad.numpy())
    for k, p in model.state_dict().items():
        out["w:" + k] = p.numpy()
    for k, p in model.named_parameters():
        out["g:" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "x_out", tuple(xo.shape), "params", sum(p.numel() for p in model.parameters()))


def main():
    ref = ref_loader.load_reference()
    torch.set_num_threads(4)
    # BASELINE.json configs 1-4 at fixture-sized batches (+ a mode-count / Nyquist case)
    run_egno(ref, "egno_n5_t8", n_balls=5, B=4, T=8, n_layers=4, num_modes=2)
    run_egno(ref, "egno_n20_t10", n_balls=20, B=2, T=10, n_layers=4, num_modes=2)
    run_egno(ref, "egno_n5_t6_m4", n_balls=5, B=3, T=6, n_layers=2, num_modes=4)   # modes == T//2+1 (Nyquist)
    run_egno(ref, "egno_n7_t10_m5", n_balls=7, B=2, T=10, n_layers=1, num_modes=5)
    run_egno_multi(ref, "egno_n5_t10_in3", n_balls=5, B=3, T=10, n_layers=2, num_modes=2, num_inputs=3, var_dt=False,
                   frames=[26, 28, 30])
    run_egno_multi(ref, "egno_n5_t8_in2_vardt", n_balls=5, B=4, T=8, n_layers=2, num_modes=2, num_inputs=2, var_dt=True,
                   frames=[25, 30])
    run_segno(ref, "segno_n5_t10", "charged", n_balls=5, B=4, T=10, frame0=30)
    run_segno(ref, "segno_n20_t10_gravity", "gravity", n_balls=20, B=2, T=10, frame0=0)
    run_segno_multi(ref, "segno_n5_t6_in3_attn", n_balls=5, B=3, T=6, frames=[24, 27, 30], agg="attn")
    run_segno_multi(ref, "segno_n5_t5_in2_sum", n_balls=5, B=4, T=5, frames=[26, 30], agg="sum")


if __name__ == "__main__":
    main()
