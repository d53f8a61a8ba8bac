"""EGNO with floating-point times: non-integral timesteps_out / timesteps_in, and dL/dtimes.

The reference embeds `timesteps.float()` (layer_no.py:8-17), so it takes any real time and its autograd returns
dL/dtimesteps through the sinusoidal embedding.  A floating-point time tensor takes nb_egno_forward_ft /
nb_egno_backward_ft (k_time_table_f, k_time_grad); int64 times keep the int64 entry points.

The reference is the float64 oracle of test_config_space.py with the times as float64 leaves.  Inside it the time
embedding is replaced by `_timestep_embedding_f64`: the same fp32-rounded times and fp32 frequencies, with the product
and sin / cos in float64, so that the time gradient it gives is not limited by fp32.
"""
from __future__ import annotations

import contextlib
import ctypes
import math
import re

import numpy as np
import pytest
import torch

import no_node_comparison_b200 as nb
from no_node_comparison_b200 import _cabi, synth
from oracle import nbody_oracle as O
from tests.helpers import rel_err
from tests.test_config_space import (EMU_MAX_NODES, TOL_EMU, TOL_GRAD, TOL_OUT, _nodes, check_case, cotangents, egno,
                                     make_inputs, make_model, weights_of)
from tests.test_input_grads import check_new_grads

CASES = [
    egno("ft_N5", 201, B=3, N=5, T=4, L=2),
    egno("ft_N20_sel3", 202, B=4, N=20, T=10, L=2, emu=False),     # k_edge_fwd_sel3 (N = 17 .. 27)
    egno("ft_N37_blocked", 203, B=2, N=37, T=4, L=1, emu=False),   # the blocked walk (N > 27)
    egno("ft_in2_T10", 204, B=2, N=5, T=10, L=2, num_inputs=2, vardt=True),
    egno("ft_in3_T10", 205, B=2, N=5, T=10, L=2, num_inputs=3, vardt=True),   # tmap 0 0 0 1 1 1 2 2 2 2
    egno("ft_no_time_conv", 206, B=3, N=5, T=6, L=2, use_time_conv=False),
    egno("ft_temb0", 207, B=3, N=5, T=4, L=2, time_emb_dim=0),
    egno("ft_temb64", 208, B=3, N=5, T=4, L=2, in_node_nf=3, time_emb_dim=64, vardt=True),
    # B = 3, N = 5, a different time row per trajectory: node k reads row k mod B, not k // N (egno.py:66,69)
    egno("ft_quirk_B3_N5", 209, B=3, N=5, T=4, L=1, vardt=True),
]


def _emu_cases():
    return [c for c in CASES if c["emu"] and _nodes(c) <= EMU_MAX_NODES]


def float_times(c):
    """Non-integral float64 times: t_out = 0.37 + 0.61 k, or per-trajectory sorted random reals (varDT, and the quirk
    case); t_in [B, L] sorted reals ending at 0.  Rounded to fp32 by the model, exactly as `.float()` does."""
    B, T = c["B"], c["T"]
    gen = torch.Generator().manual_seed(3000 + c["seed"])
    if c["vardt"]:
        t_out = torch.sort(0.2 + 2 * T * torch.rand(B, T, generator=gen, dtype=torch.float64), dim=1).values
    else:
        t_out = (0.37 + 0.61 * torch.arange(1, T + 1, dtype=torch.float64))[None].repeat(B, 1)
    t_in = None
    if c["num_inputs"] > 1:
        steps = 0.3 + torch.rand(B, c["num_inputs"] - 1, generator=gen, dtype=torch.float64)
        t_in = torch.cat([-steps.flip(1).cumsum(1).flip(1), torch.zeros(B, 1, dtype=torch.float64)], dim=1)
    return t_out, t_in


# ----------------------------------------------------------------------------------------------------- the oracle
def _timestep_embedding_f64(timesteps, dim, max_positions=10000):
    """O.timestep_embedding (layer_no.py:8-17) with the fp32-rounded times (`timesteps.float()`) and the fp32
    frequencies multiplied and passed through sin / cos in float64."""
    half = dim // 2
    scale = math.log(max_positions) / (half - 1)
    freq = torch.exp(torch.arange(half, dtype=torch.float32, device=timesteps.device) * -scale).double()
    arg = timesteps.float().double()[:, :, None] * freq[None, None, :]
    return torch.cat([torch.sin(arg), torch.cos(arg)], dim=-1)


@contextlib.contextmanager
def _float64_time_embedding():
    orig = O.timestep_embedding
    O.timestep_embedding = _timestep_embedding_f64
    try:
        yield
    finally:
        O.timestep_embedding = orig


def oracle_ft(c, w, inp, G, t_out, t_in):
    """Outputs and gradients (float64, CPU) of every input, the times included, and the parameter leaves.

    time_emb_dim = 0: the oracle's broadcast reshape needs a time width, so it runs with four time features whose
    embedding columns are zero.  That leaves the outputs and every other gradient as they are, gives the times the
    zero gradient of an unused input, and the extra columns' weight gradient is dropped with them."""
    f64 = lambda t: t.double()
    leaf = lambda t: f64(t).detach().requires_grad_(True)
    p = {k: leaf(t) for k, t in w.items()}
    x, v, to = leaf(inp["x"]), leaf(inp["v"]), leaf(t_out)
    D = c["time_emb_dim"]
    pw = dict(p)
    if D == 0:
        D = 4
        pw["embedding.weight"] = torch.cat([p["embedding.weight"], torch.zeros(64, D, dtype=torch.float64)], dim=1)
    kw = dict(n_layers=c["L"], num_timesteps=c["T"], time_emb_dim=D)
    single = c["num_inputs"] == 1
    with _float64_time_embedding():
        if single:
            nodes, ea, lm = leaf(inp["nodes"]), leaf(inp["ea"]), leaf(inp["lm"])
            xo, vo, ho = O.egno_forward(pw, x, nodes, inp["row"], inp["col"], ea, v, lm, to,
                                        use_time_conv=c["use_time_conv"], **kw)
        else:
            ti = leaf(t_in)
            xo, vo, ho = O.egno_forward_multi(pw, x, f64(inp["nodes"]), inp["row"], inp["col"], f64(inp["ea"]), v,
                                              f64(inp["lm"]), ti, to, **kw)
    ((xo * f64(G["x"])).sum() + (vo * f64(G["v"])).sum() + (ho * f64(G["h"])).sum()).backward()
    grad = lambda t: t.grad if t.grad is not None else torch.zeros(t.shape, dtype=torch.float64)   # an unused leaf
    out = dict(x=xo.detach(), v=vo.detach(), h=ho.detach(), gx=x.grad, gv=v.grad, gt_out=grad(to))
    if single:
        out.update(gnodes=grad(nodes), gea=grad(ea), glm=grad(lm))
    else:
        out["gt_in"] = grad(ti)
    return out, p


def check_time_grads(c, got, ref, tol, label):
    for k in ("gt_out", "gt_in"):
        if k not in ref:
            continue
        assert tuple(got[k].shape) == tuple(ref[k].shape), (k, got[k].shape, ref[k].shape)
        if c["time_emb_dim"] == 0:
            assert not bool(got[k].any()), k
            continue
        e = rel_err(got[k], ref[k])
        print(f"{label} {c['name']}: {k} rel err {e:.1e} (bar {tol:.0e})")
        assert e < tol, (c["name"], k, e)


def check_all(c, got, m, ref, p, tol_out, tol_grad, w, inp, G, label):
    check_case(c, got, m, ref, p, tol_out, tol_grad, w, inp, G, label)
    if c["num_inputs"] == 1:
        check_new_grads(c, got, ref, tol_grad, w, inp, G, label)
    check_time_grads(c, got, ref, tol_grad, label)


# ----------------------------------------------------------------------------------------------------- CPU tier
def emu_run_ft(c, m, inp, G, t_out, t_in):
    """nb_egno_forward_ft, then nb_egno_backward_ft with every gradient requested, through the host emulator."""
    from tests import emu_harness as E

    L = E.lib()
    params = E.flat_params({k: t.detach().numpy() for k, t in m.named_parameters()}, [k for k, _ in m.named_parameters()])
    n = lambda t: E.f32(t.numpy())
    nin = c["num_inputs"]
    cfg = E.cabi.NbEgnoConfig(B=c["B"], N=c["N"], T=c["T"], n_layers=c["L"],
                             num_modes=m.num_modes if c["use_time_conv"] else 1, in_node_nf=c["in_node_nf"],
                             in_edge_nf=c["in_edge_nf"], time_emb_dim=c["time_emb_dim"],
                             use_time_conv=int(c["use_time_conv"]), num_inputs=nin)
    Nn, n0 = cfg.T * cfg.B * cfg.N, cfg.B * cfg.N
    x, nodes, ea, v, lm = n(inp["x"]), n(inp["nodes"]), n(inp["ea"]), n(inp["v"]), n(inp["lm"])
    to = n(t_out)
    ti = None if t_in is None else n(t_in)
    outs = [np.zeros((Nn, k), np.float32) for k in (3, 3, 64)]
    saved = np.zeros(L.nb_egno_saved_floats(ctypes.byref(cfg)), np.float32)
    ws = np.zeros(L.nb_egno_workspace_floats(ctypes.byref(cfg), 2), np.float32)
    E.check(L.nb_egno_forward_ft(ctypes.byref(cfg), E.ptr(params), E.ptr(x), E.ptr(nodes), E.ptr(ea), E.ptr(v), E.ptr(lm),
                                 E.ptr(to), E.ptr(ti), *[E.ptr(o) for o in outs], E.ptr(saved), E.ptr(ws), None))
    lead = (nin,) if nin > 1 else ()
    gp = np.full(params.size, np.nan, np.float32)
    gx, gv = (np.full(lead + (n0, 3), np.nan, np.float32) for _ in range(2))
    gt_out = np.full(to.shape, np.nan, np.float32)
    gt_in = None if ti is None else np.full(ti.shape, np.nan, np.float32)
    single = nin == 1
    gnodes = np.full(nodes.shape, np.nan, np.float32) if single else None
    gea = np.full(ea.shape, np.nan, np.float32) if single and ea.size else None
    glm = np.full(lm.shape, np.nan, np.float32) if single else None
    ws2 = np.zeros(L.nb_egno_workspace_floats(ctypes.byref(cfg), 1), np.float32)
    iws = np.zeros(L.nb_egno_input_grad_workspace_floats(ctypes.byref(cfg)), np.float32)
    E.check(L.nb_egno_backward_ft(ctypes.byref(cfg), E.ptr(params), E.ptr(nodes), E.ptr(ea), E.ptr(lm), E.ptr(to), E.ptr(ti),
                                  E.ptr(saved), E.ptr(n(G["x"])), E.ptr(n(G["v"])), E.ptr(n(G["h"])), E.ptr(gp), E.ptr(gx),
                                  E.ptr(gv), E.ptr(gnodes), E.ptr(gea), E.ptr(glm), E.ptr(gt_out), E.ptr(gt_in), E.ptr(ws2),
                                  E.ptr(iws), None))
    off = 0
    for _, q in m.named_parameters():
        q.grad = torch.tensor(gp[off:off + q.numel()]).view_as(q)
        off += q.numel()
    res = dict(x=outs[0], v=outs[1], h=outs[2], gx=gx, gv=gv, gt_out=gt_out)
    if single:
        res.update(gnodes=gnodes, gea=gea if gea is not None else np.zeros(ea.shape, np.float32), glm=glm)
    else:
        res["gt_in"] = gt_in
    return {k: torch.tensor(a) for k, a in res.items()}


@pytest.mark.parametrize("c", _emu_cases(), ids=lambda c: c["name"])
def test_emulated_float_times_vs_float64_oracle(c):
    """The new entry points through the host emulator (fp32 SIMT kernels) against float64 autograd, at 2e-5."""
    m = make_model(c, "cpu")
    w = weights_of(m)
    inp = make_inputs(c)
    G = cotangents(c)
    t_out, t_in = float_times(c)
    ref, p = oracle_ft(c, w, inp, G, t_out, t_in)
    got = emu_run_ft(c, m, inp, G, t_out, t_in)
    check_all(c, got, m, ref, p, TOL_EMU, TOL_EMU, w, inp, G, "emulator")


def test_the_quirk_case_separates_k_mod_b_from_k_div_n():
    """In the quirk case the two row maps give different embeddings and time gradients, so a kernel that used k // N
    could not pass the oracle comparisons above."""
    c = next(c for c in CASES if c["name"] == "ft_quirk_B3_N5")
    B, N = c["B"], c["N"]
    t_out, _ = float_times(c)
    assert all(not torch.equal(t_out[i], t_out[j]) for i in range(B) for j in range(i + 1, B))
    k = torch.arange(B * N)
    assert not torch.equal(k % B, k // N)


# ----------------------------------------------------------------------------------------------------- GPU tier
def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    return torch.device("cuda:0")


def cuda_run(c, m, inp, G, t_out, t_in, want_inputs=True, want_t=True):
    """Module forward + backward; t_out / t_in are the caller's tensors (any dtype), leaves requiring grad if want_t."""
    d = _dev()
    single = c["num_inputs"] == 1
    x = inp["x"].to(d).requires_grad_(True)
    v = inp["v"].to(d).requires_grad_(True)
    nodes = inp["nodes"].to(d).requires_grad_(want_inputs and single)
    ea = inp["ea"].to(d).requires_grad_(want_inputs and single)
    lm = inp["lm"].to(d).requires_grad_(want_inputs and single)
    to = t_out.to(d).requires_grad_(want_t and t_out.is_floating_point())
    ti = None if t_in is None else t_in.to(d).requires_grad_(want_t and t_in.is_floating_point())
    xo, vo, ho = m(x, nodes, [inp["row"].to(d), inp["col"].to(d)], ea, v=v, loc_mean=lm, timesteps_in=ti,
                   timesteps_out=to)
    ((xo * G["x"].to(d)).sum() + (vo * G["v"].to(d)).sum() + (ho * G["h"].to(d)).sum()).backward()
    cpu = lambda t: t.detach().cpu()
    got = dict(x=cpu(xo), v=cpu(vo), h=cpu(ho), gx=cpu(x.grad), gv=cpu(v.grad))
    if want_inputs and single:
        got.update(gnodes=cpu(nodes.grad), gea=cpu(ea.grad), glm=cpu(lm.grad))
    if to.requires_grad:
        got["gt_out"] = cpu(to.grad)
        assert to.grad.dtype == to.dtype and to.grad.shape == to.shape
    if ti is not None and ti.requires_grad:
        got["gt_in"] = cpu(ti.grad)
        assert ti.grad.dtype == ti.dtype and ti.grad.shape == ti.shape
    got["params"] = {k: cpu(q.grad).clone() for k, q in m.named_parameters() if q.grad is not None}
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=lambda c: c["name"])
def test_float_times_cuda_vs_float64_oracle(c):
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    m = make_model(c, d)
    w = weights_of(m)
    t_out, t_in = float_times(c)
    ref, p = oracle_ft(c, w, inp, G, t_out, t_in)
    got = cuda_run(c, m, inp, G, t_out, t_in)
    check_all(c, got, m, ref, p, TOL_OUT, TOL_GRAD, w, inp, G, "cuda")


_BITWISE = [egno("ft_cfg3_full", 101, B=256, N=20, T=10, L=4), egno("ft_N5_packed", 103, B=100, N=5, T=8, L=4),
            egno("ft_N37_blocked_bw", 104, B=2, N=37, T=4, L=2),
            egno("ft_in3_bw", 105, B=8, N=20, T=10, L=2, num_inputs=3, vardt=True)]


def _assert_same(a, b, keys):
    for k in keys:
        assert torch.equal(a[k], b[k]), k
    assert a["params"].keys() == b["params"].keys()
    for k in a["params"]:
        assert torch.equal(a["params"][k], b["params"][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("c", _BITWISE, ids=lambda c: c["name"])
def test_integral_float_times_equal_int64_times_bitwise(c):
    """The same integral times as int64 and as float32 (k_time_table vs k_time_table_f): outputs, input gradients and
    every parameter gradient bit for bit."""
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    t_out, t_in = inp["t_out"], inp["t_in"]
    a = cuda_run(c, make_model(c, d), inp, G, t_out, t_in, want_t=False)
    b = cuda_run(c, make_model(c, d), inp, G, t_out.float(), None if t_in is None else t_in.float(), want_t=True)
    keys = ["x", "v", "h", "gx", "gv"] + (["gnodes", "gea", "glm"] if c["num_inputs"] == 1 else [])
    _assert_same(a, b, keys)


@pytest.mark.gpu
@pytest.mark.parametrize("c", _BITWISE, ids=lambda c: c["name"])
def test_requesting_time_grads_changes_nothing_else_and_is_deterministic(c):
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    t_out, t_in = float_times(c)
    a = cuda_run(c, make_model(c, d), inp, G, t_out, t_in, want_t=False)
    b, b2 = (cuda_run(c, make_model(c, d), inp, G, t_out, t_in, want_t=True) for _ in range(2))
    keys = ["x", "v", "h", "gx", "gv"] + (["gnodes", "gea", "glm"] if c["num_inputs"] == 1 else [])
    _assert_same(a, b, keys)
    for k in ("gt_out", "gt_in"):
        if k in b:
            assert torch.equal(b[k], b2[k]), k
            assert bool(torch.isfinite(b[k]).all()), k


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.gpu
def test_launches_of_int64_and_float_time_steps():
    """cfg3 forward + backward: int64 times launch what the parent launched (62, no new kernel); float times without
    time gradients the same count with k_time_table_f for k_time_table; time gradients add one k_time_grad."""
    c = egno("ft_cfg3_full", 101, B=256, N=20, T=10, L=4)
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    m = make_model(c, d)
    lib = nb.load_library()
    t_f, _ = float_times(c)
    arms = dict(int64=(inp["t_out"], False), float=(t_f, False), float_grad=(t_f, True))
    counts, names = {}, {}
    for arm, (t, want_t) in arms.items():
        run = lambda: cuda_run(c, m, inp, G, t, None, want_inputs=False, want_t=want_t)
        run()
        torch.cuda.synchronize()
        n0 = lib.nb_launch_count()
        run()
        counts[arm] = lib.nb_launch_count() - n0
        names[arm] = _kernel_names(run)
        print(arm, counts[arm], sorted({n for n in names[arm] if "k_time" in n}))
    has = lambda arm, k: any(re.search(rf"\b{k}\b", n) for n in names[arm])
    assert counts["int64"] == 62, counts
    assert has("int64", "k_time_table") and not has("int64", "k_time_table_f") and not has("int64", "k_time_grad")
    assert counts["float"] == 62 and has("float", "k_time_table_f") and not has("float", "k_time_table")
    assert not has("float", "k_time_grad")
    assert counts["float_grad"] == 63 and has("float_grad", "k_time_grad")


@pytest.mark.gpu
def test_graphed_float_time_training_step_matches_eager():
    """Learnable fractional output times, trained with the weights: GraphedStep (forward, backward with dL/dtimes,
    Adam, captured in one CUDA graph) follows the eager steps bit for bit."""
    c = egno("ft_graph", 211, B=16, N=20, T=10, L=2)
    d = _dev()
    inp = make_inputs(c)
    t0, _ = float_times(c)
    ins = dict(x=inp["x"].to(d), nodes=inp["nodes"].to(d), ea=inp["ea"].to(d), v=inp["v"].to(d), lm=inp["lm"].to(d))
    edges = [inp["row"].to(d), inp["col"].to(d)]
    tgt = (inp["x"].repeat(c["T"], 1) + 0.05 * torch.randn(c["T"] * 16 * 20, 3, generator=torch.Generator().manual_seed(2))).to(d)
    losses, times = {}, {}
    for mode in ("eager", "graph"):
        m = make_model(c, d)
        t_out = torch.nn.Parameter(t0.float().to(d))
        opt = torch.optim.Adam([{"params": m.parameters()}, {"params": [t_out], "lr": 1e-2}], lr=1e-3, capturable=True)

        def fn(x, nodes, ea, v, lm):
            xo, _, _ = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
            return ((xo - tgt) ** 2).mean()

        out = []
        if mode == "graph":
            step = nb.GraphedStep(fn, ins, opt, warmup=3)
            for _ in range(4):
                out.append(float(step(**ins)))
        else:
            for _ in range(7):
                opt.zero_grad(set_to_none=True)
                loss = fn(**ins)
                loss.backward()
                opt.step()
                out.append(float(loss.detach()))
        losses[mode] = out
        times[mode] = t_out.detach().cpu().clone()
    assert losses["graph"] == losses["eager"][3:], losses
    assert torch.equal(times["graph"], times["eager"])
    assert not torch.equal(times["eager"], t0.float())


# ---- guard bands around the raw entry points
def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,T,nin", [(3, 20, 10, 1), (2, 29, 4, 1), (3, 20, 10, 3), (2, 5, 6, 2)])
def test_egno_ft_entry_points_never_write_outside_their_buffers(B, N, T, nin):
    from tests.test_gpu_guards import SENT, Arena
    d = _dev()
    lib = nb.load_library()
    row, col = synth.canonical_edges(B, N)
    s = synth.sample_state("charged", B, N, seed=7)
    x, nodes, ea, v, lm = [t.contiguous() for t in synth.egno_features(s["loc"], s["vel"], s["charges"], row, col)]
    if nin > 1:
        x, nodes, ea, v, lm = [t[None].repeat(nin, *([1] * t.dim())).contiguous() for t in (x, nodes, ea, v, lm)]
    x, nodes, ea, v, lm = [t.to(d) for t in (x, nodes, ea, v, lm)]
    cfg = _cabi.NbEgnoConfig(B, N, T, 2, 2, 2, 2, 32, 1, nin)
    npar = lib.nb_egno_param_count(ctypes.byref(cfg))
    params = (0.1 * torch.randn(npar, generator=torch.Generator().manual_seed(1))).to(d)
    ts = (0.37 + 0.61 * torch.arange(1, T + 1, dtype=torch.float32))[None].repeat(B, 1).to(d).contiguous()
    ts_in = (-0.45 * torch.arange(nin - 1, -1, -1, dtype=torch.float32))[None].repeat(B, 1).to(d).contiguous() if nin > 1 else None
    Nn, n0, E0 = T * B * N, B * N, B * N * (N - 1)
    single = nin == 1
    lead = 1 if single else nin
    st = ctypes.c_void_p(torch.cuda.current_stream(d).cuda_stream)
    sizes = dict(x_out=Nn * 3, v_out=Nn * 3, h_out=Nn * 64, saved=lib.nb_egno_saved_floats(ctypes.byref(cfg)),
                 ws_f=lib.nb_egno_workspace_floats(ctypes.byref(cfg), 2), ws_b=lib.nb_egno_workspace_floats(ctypes.byref(cfg), 1),
                 grad=npar, gx_in=lead * n0 * 3, gv_in=lead * n0 * 3, g_t=B * T)
    if single:
        sizes.update(iws=lib.nb_egno_input_grad_workspace_floats(ctypes.byref(cfg)), g_nodes=n0 * 2, g_ef=E0 * 2, g_lm=n0 * 3)
    else:
        sizes.update(g_t_in=B * nin)
    A = Arena(sizes, d)
    opt = lambda k: A.ptr(k) if k in sizes else None
    rc = lib.nb_egno_forward_ft(ctypes.byref(cfg), _p(params), _p(x), _p(nodes), _p(ea), _p(v), _p(lm), _p(ts), _p(ts_in),
                                A.ptr("x_out"), A.ptr("v_out"), A.ptr("h_out"), A.ptr("saved"), A.ptr("ws_f"), st)
    assert rc == 0, lib.nb_last_error()
    g = torch.Generator().manual_seed(2)
    Gx, Gv, Gh = [torch.randn(Nn, k, generator=g).to(d) for k in (3, 3, 64)]
    rc = lib.nb_egno_backward_ft(ctypes.byref(cfg), _p(params), _p(nodes), _p(ea), _p(lm), _p(ts), _p(ts_in), A.ptr("saved"),
                                 _p(Gx), _p(Gv), _p(Gh), A.ptr("grad"), A.ptr("gx_in"), A.ptr("gv_in"), opt("g_nodes"),
                                 opt("g_ef"), opt("g_lm"), A.ptr("g_t"), opt("g_t_in"), A.ptr("ws_b"), opt("iws"), st)
    assert rc == 0, lib.nb_last_error()
    torch.cuda.synchronize()
    assert A.guards_intact()
    for k in sizes:
        if k in ("saved", "ws_f", "ws_b", "iws"):
            continue
        assert not bool((A.view(k) == SENT).any()), k
        assert bool(torch.isfinite(A.view(k)).all()), k
