"""Gradients of EGNO / SEGNO with respect to their node features, edge features and (EGNO) loc_mean.

The single-input forward of both models backpropagates to every input, as the reference's plain-PyTorch modules do:
EGNO to h, edge_fea and loc_mean besides x and v; SEGNO.forward to his and edge_attr; SEGNO.forward_step to h and
edge_attr.  This is what unrolled (multi-call) training needs: the next call's features are the previous call's
predictions run through the featurisation.

The oracle of test_config_space.py, extended here so that the node features, edge features, loc_mean and his are float64
leaves too, is the reference.  Requesting the new gradients must not change anything else: outputs, dL/dx, dL/dv and
every parameter gradient stay bitwise equal, and a step without them launches neither the EGRAD instantiations of the
edge backward kernels nor the new reduction kernels.
"""
from __future__ import annotations

import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import no_node_comparison_b200 as nb
from no_node_comparison_b200 import _cabi, synth
from oracle import nbody_oracle as O
from tests.helpers import rel_err
from tests.test_config_space import (CASES, ENVELOPE, TOL_EMU, TOL_GRAD, TOL_OUT, _emu_cases, check_case, cotangents,
                                     egno, make_inputs, make_model, segno, weights_of)

# full-size shapes, like test_gpu_parity.py's full-batch cases: BASELINE.json configs[2] and the 100-body system
FULL = [egno("egno_cfg3_full", 101, B=256, N=20, T=10, L=4, emu=False),
        # one layer, like test_gpu_parity.py's 100-body case: with 4 layers, T = 10 and the 20x temporal convolution
        # the forward's x sits at 1.7e-4 of float64 (fp32 oracle: 3.2e-6), outside the 1e-4 output bar this file reuses
        egno("egno_N100_B4", 102, B=4, N=100, T=3, L=1, emu=False)]
GPU_CASES = [c for c in CASES if c["model"] == "segno" or c["num_inputs"] == 1] + FULL
NEW = {"egno": ("gnodes", "gea", "glm"), "segno": ("ghis", "gea")}


def _single_input(cases):
    return [c for c in cases if c["model"] == "segno" or c["num_inputs"] == 1]


# ----------------------------------------------------------------------------------------------------- the oracle
def oracle_inputs(c, w, inp, G, dtype=torch.float64, device="cpu"):
    """Outputs, gradients of every input and parameter leaves (with .grad, on the CPU) of the float64 oracle."""
    dv = lambda t: t.to(device=device, dtype=dtype)
    leaf = lambda t: dv(t).requires_grad_(True)
    p = {k: leaf(t.detach()) for k, t in w.items()}
    x, v = leaf(inp["x"]), leaf(inp["v"])
    ea = leaf(inp["ea"])
    row, col = inp["row"].to(device), inp["col"].to(device)
    if c["model"] == "egno":
        nodes, lm = leaf(inp["nodes"]), leaf(inp["lm"])
        xo, vo, ho = O.egno_forward(p, x, nodes, row, col, ea, v, lm, inp["t_out"].to(device), n_layers=c["L"],
                                    num_timesteps=c["T"], time_emb_dim=c["time_emb_dim"],
                                    use_time_conv=c["use_time_conv"])
    else:
        his = leaf(inp["his"])
        xo, ho, vo = O.segno_forward(p, his, x, row, col, v, ea, c["T"], recurrent=c["recurrent"],
                                     coords_weight=c["coords_weight"])
    ((xo * dv(G["x"])).sum() + (vo * dv(G["v"])).sum() + (ho * dv(G["h"])).sum()).backward()
    cpu = lambda t: None if t is None else t.detach().cpu()
    grad = lambda t: cpu(t.grad) if t.grad is not None else torch.zeros(t.shape, dtype=dtype)   # an input left unused
    out = dict(x=cpu(xo), v=cpu(vo), h=cpu(ho), gx=cpu(x.grad), gv=cpu(v.grad), gea=grad(ea))
    if c["model"] == "egno":
        out.update(gnodes=grad(nodes), glm=grad(lm))
    else:
        out.update(ghis=grad(his))
    pc = {}
    for k, t in p.items():
        pc[k] = t.detach().cpu().requires_grad_(True)
        pc[k].grad = cpu(t.grad)
    return out, pc


def check_new_grads(c, got, ref, tol, w=None, inp=None, G=None, label=""):
    if c["envelope"]:   # the deep case: a multiple of the fp32 oracle's own distance from float64
        r32, _ = oracle_inputs(c, w, inp, G, dtype=torch.float32)
        tol = max(tol, ENVELOPE * max(rel_err(r32[k], ref[k]) for k in NEW[c["model"]] if ref[k].numel()))
    errs = {}
    for k in NEW[c["model"]]:
        assert tuple(got[k].shape) == tuple(ref[k].shape), (k, got[k].shape, ref[k].shape)
        errs[k] = rel_err(got[k], ref[k]) if ref[k].numel() else 0.0
    print(f"{label} {c['name']}: new input gradients " + " ".join(f"{k}={e:.1e}" for k, e in errs.items()) + f" (bar {tol:.0e})")
    for k, e in errs.items():
        assert e < tol, (c["name"], k, errs)


# ----------------------------------------------------------------------------------------------------- CPU tier
def _emu_run_ex(c, m, inp, G):
    """The emulated C ABI: forward, then nb_*_backward_ex with every new gradient requested."""
    from tests import emu_harness as E

    L = E.lib()
    order = [k for k, _ in m.named_parameters()]
    params = E.flat_params({k: t.detach().numpy() for k, t in m.named_parameters()}, order)
    n = lambda t: None if t is None else E.f32(t.numpy())
    if c["model"] == "egno":
        cfg = E.cabi.NbEgnoConfig(B=c["B"], N=c["N"], T=c["T"], n_layers=c["L"],
                                 num_modes=m.num_modes if c["use_time_conv"] else 1, in_node_nf=c["in_node_nf"],
                                 in_edge_nf=c["in_edge_nf"], time_emb_dim=c["time_emb_dim"],
                                 use_time_conv=int(c["use_time_conv"]), num_inputs=1)
        Nn = cfg.T * cfg.B * cfg.N
        x, nodes, ea, v, lm = n(inp["x"]), n(inp["nodes"]), n(inp["ea"]), n(inp["v"]), n(inp["lm"])
        t_out = np.ascontiguousarray(inp["t_out"].numpy().astype(np.int64))
        outs = [np.zeros((Nn, k), np.float32) for k in (3, 3, 64)]
        saved = np.zeros(L.nb_egno_saved_floats(ctypes.byref(cfg)), np.float32)
        ws = np.zeros(L.nb_egno_workspace_floats(ctypes.byref(cfg), 0), np.float32)
        E.check(L.nb_egno_forward(ctypes.byref(cfg), E.ptr(params), E.ptr(x), E.ptr(nodes), E.ptr(ea), E.ptr(v), E.ptr(lm),
                                  E.ptr(t_out), None, *[E.ptr(o) for o in outs], E.ptr(saved), E.ptr(ws), None))
        gp = np.full(params.size, np.nan, np.float32)
        gx, gv, glm = (np.full((cfg.B * cfg.N, 3), np.nan, np.float32) for _ in range(3))
        gnodes = np.full(nodes.shape, np.nan, np.float32)
        gea = np.full(ea.shape, np.nan, np.float32)
        ws2 = np.zeros(L.nb_egno_workspace_floats(ctypes.byref(cfg), 1), np.float32)
        iws = np.zeros(L.nb_egno_input_grad_workspace_floats(ctypes.byref(cfg)), np.float32)
        E.check(L.nb_egno_backward_ex(ctypes.byref(cfg), E.ptr(params), E.ptr(nodes), E.ptr(ea), E.ptr(lm), E.ptr(t_out), None,
                                      E.ptr(saved), E.ptr(n(G["x"])), E.ptr(n(G["v"])), E.ptr(n(G["h"])), E.ptr(gp), E.ptr(gx),
                                      E.ptr(gv), E.ptr(gnodes), E.ptr(gea) if gea.size else None, E.ptr(glm), E.ptr(ws2),
                                      E.ptr(iws), None))
        res = dict(x=outs[0], v=outs[1], h=outs[2], gx=gx, gv=gv, gnodes=gnodes, gea=gea, glm=glm)
    else:
        cfg = E.cabi.NbSegnoConfig(B=c["B"], N=c["N"], T=c["T"], in_node_nf=c["in_node_nf"], in_edge_nf=c["in_edge_nf"],
                                  recurrent=int(c["recurrent"]), coords_weight=c["coords_weight"], h_given=0)
        Nn = cfg.B * cfg.N
        his, x, v, ea = n(inp["his"]), n(inp["x"]), n(inp["v"]), n(inp["ea"])
        outs = [np.zeros((Nn, k), np.float32) for k in (3, 64, 3)]
        saved = np.zeros(L.nb_segno_saved_floats(ctypes.byref(cfg)), np.float32)
        ws = np.zeros(L.nb_segno_workspace_floats(ctypes.byref(cfg), 0), np.float32)
        E.check(L.nb_segno_forward(ctypes.byref(cfg), E.ptr(params), E.ptr(his), E.ptr(x), E.ptr(v), E.ptr(ea),
                                   *[E.ptr(o) for o in outs], E.ptr(saved), E.ptr(ws), None))
        gp = np.full(params.size, np.nan, np.float32)
        gx, gv = (np.full((Nn, 3), np.nan, np.float32) for _ in range(2))
        ghis = np.full(his.shape, np.nan, np.float32)
        gea = np.full(ea.shape, np.nan, np.float32)
        ws2 = np.zeros(L.nb_segno_workspace_floats(ctypes.byref(cfg), 1), np.float32)
        iws = np.zeros(L.nb_segno_input_grad_workspace_floats(ctypes.byref(cfg)), np.float32)
        E.check(L.nb_segno_backward_ex(ctypes.byref(cfg), E.ptr(params), E.ptr(his), E.ptr(ea), E.ptr(saved), E.ptr(n(G["x"])),
                                       E.ptr(n(G["h"])), E.ptr(n(G["v"])), E.ptr(gp), E.ptr(gx), E.ptr(gv), None, E.ptr(ghis),
                                       E.ptr(gea) if gea.size else None, E.ptr(ws2), E.ptr(iws), None))
        res = dict(x=outs[0], h=outs[1], v=outs[2], gx=gx, gv=gv, ghis=ghis, gea=gea)
    off = 0
    for _, q in m.named_parameters():
        q.grad = torch.tensor(gp[off:off + q.numel()]).view_as(q)
        off += q.numel()
    return {k: torch.tensor(a) for k, a in res.items()}


@pytest.mark.parametrize("c", _single_input(_emu_cases()), ids=lambda c: c["name"])
def test_emulated_input_grads_vs_float64_oracle(c):
    """nb_egno_backward_ex / nb_segno_backward_ex through the host emulator (fp32 SIMT kernels, EGRAD instantiation of
    k_edge_bwd) against float64 autograd; everything else the entry points return is held to the same bar."""
    m = make_model(c, "cpu")
    w = weights_of(m)
    inp = make_inputs(c)
    G = cotangents(c)
    ref, p = oracle_inputs(c, w, inp, G)
    got = _emu_run_ex(c, m, inp, G)
    check_case(c, got, m, ref, p, TOL_EMU, TOL_EMU, w, inp, G, "emulator")
    check_new_grads(c, got, ref, TOL_EMU, w, inp, G, "emulator")


# registers / stack bytes / static shared memory of the edge backward kernels without input gradients, as a build of the
# parent commit reports them (cuobjdump -res-usage; its ptxas -v said 0 / 0 spill bytes for the whole-graph walk and
# k_edge_bwd, 16 / 24 for the blocked walk).  The EGRAD = false instantiations must keep them.
_PARENT_RES = {
    "_Z14k_edge_bwd_selILb0ELb0EEv13NbEdgeBwdArgs": dict(REG=128, STACK=120, SHARED=1024, LOCAL=0),
    "_Z14k_edge_bwd_selILb1ELb0EEv13NbEdgeBwdArgs": dict(REG=128, STACK=136, SHARED=1024, LOCAL=0),
    "_Z10k_edge_bwdILb0EEv13NbEdgeBwdArgs": dict(REG=255, STACK=0, SHARED=1024, LOCAL=0),
}
_EGRAD = ["_Z14k_edge_bwd_selILb0ELb1EEv13NbEdgeBwdArgs", "_Z14k_edge_bwd_selILb1ELb1EEv13NbEdgeBwdArgs",
          "_Z10k_edge_bwdILb1EEv13NbEdgeBwdArgs"]


def test_edge_backward_without_input_grads_keeps_the_parent_resources():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.isfile(exe):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([exe, "-res-usage", nb.build_library()], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    res = {}
    for fn, line in re.findall(r"Function (\S+):\s*\n\s*(REG:.*)", out.stdout):
        res[fn] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
    for fn, want in _PARENT_RES.items():
        assert fn in res, fn
        assert res[fn] == want, (fn, res[fn], want)
    for fn in _EGRAD:
        assert fn in res, f"no EGRAD instantiation {fn} in the library"
        print(fn, res[fn])


def test_multi_input_models_refuse_the_new_input_gradients():
    """Multi-input EGNO and SEGNO keep raising for node / edge features; EGNO now also refuses a loc_mean that requires
    grad instead of returning no gradient for it."""
    B, N, T, nin = 2, 5, 4, 2
    row, col = synth.canonical_edges(B, N)
    m = nb.EGNO(n_layers=1, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_timesteps=T, num_inputs=nin)
    E0 = B * N * (N - 1)
    base = dict(x=torch.zeros(nin, B * N, 3), h=torch.zeros(nin, B * N, 2), edge_fea=torch.zeros(nin, E0, 2),
                v=torch.zeros(nin, B * N, 3), loc_mean=torch.zeros(nin, B * N, 3))
    for k in ("h", "edge_fea", "loc_mean"):
        a = dict(base)
        a[k] = a[k].clone().requires_grad_(True)
        with pytest.raises(ValueError, match="not implemented"):
            m(a["x"], a["h"], [row, col], a["edge_fea"], v=a["v"], loc_mean=a["loc_mean"],
              timesteps_in=torch.zeros(B, nin, dtype=torch.long), timesteps_out=torch.ones(B, T, dtype=torch.long))
    s = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, multiple_agg='sum')
    for k in ("his", "edge_attr"):
        his, ea = torch.zeros(B * N, nin, 1), torch.zeros(E0, 2)
        if k == "his":
            his.requires_grad_(True)
        else:
            ea.requires_grad_(True)
        with pytest.raises(ValueError, match="not implemented"):
            s(his, torch.zeros(B * N, nin, 3), [row, col], torch.zeros(B * N, nin, 3), ea, T=3, in_steps=torch.tensor([0, 2]))


# ----------------------------------------------------------------------------------------------------- GPU tier
def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    return torch.device("cuda:0")


def _cuda_run(c, m, inp, G, want=True):
    d = _dev()
    x = inp["x"].to(d).requires_grad_(True)
    v = inp["v"].to(d).requires_grad_(True)
    ea = inp["ea"].to(d).requires_grad_(want)
    edges = [inp["row"].to(d), inp["col"].to(d)]
    if c["model"] == "egno":
        nodes = inp["nodes"].to(d).requires_grad_(want)
        lm = inp["lm"].to(d).requires_grad_(want)
        xo, vo, ho = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=inp["t_out"].to(d))
    else:
        his = inp["his"].to(d).requires_grad_(want)
        xo, ho, vo = m(his, x, edges, v, ea, T=c["T"])
    ((xo * G["x"].to(d)).sum() + (vo * G["v"].to(d)).sum() + (ho * G["h"].to(d)).sum()).backward()
    got = dict(x=xo.detach().cpu(), v=vo.detach().cpu(), h=ho.detach().cpu(), gx=x.grad.cpu(), gv=v.grad.cpu())
    if want:
        got["gea"] = ea.grad.cpu()
        if c["model"] == "egno":
            got.update(gnodes=nodes.grad.cpu(), glm=lm.grad.cpu())
        else:
            got["ghis"] = his.grad.cpu()
    return got


def _oracle_device(c):
    return "cuda:0" if c["name"] in ("egno_cfg3_full", "egno_N100_B4") else "cpu"


@pytest.mark.gpu
@pytest.mark.parametrize("c", GPU_CASES, ids=lambda c: c["name"])
def test_input_grads_cuda_vs_float64_oracle(c):
    """Every single-input case of the configuration table plus two full-size shapes: the new gradients at the 1e-3 bar
    (the deep case under the fp32 envelope), everything else as test_config_space.py holds it."""
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    m = make_model(c, d)
    w = weights_of(m)
    ref, p = oracle_inputs(c, w, inp, G, device=_oracle_device(c))
    fused_modes = (1, 0) if c["model"] == "segno" and c["N"] <= 27 else (None,)
    lib = nb.load_library()
    for fused in fused_modes:
        if fused is not None:
            assert lib.nb_set_segno_fused(fused) == 0
        try:
            m.zero_grad(set_to_none=True)
            got = _cuda_run(c, m, inp, G)
            check_case(c, got, m, ref, p, TOL_OUT, TOL_GRAD, w, inp, G, f"cuda fused={fused}")
            check_new_grads(c, got, ref, TOL_GRAD, w, inp, G, f"cuda fused={fused}")
        finally:
            lib.nb_set_segno_fused(1)


_UNCHANGED = [egno("egno_cfg3_full", 101, B=256, N=20, T=10, L=4), egno("egno_N5_packed", 103, B=100, N=5, T=8, L=4),
              egno("egno_N37_blocked", 104, B=2, N=37, T=4, L=2), segno("segno_cfg4", 105, B=100, N=20, T=10)]


@pytest.mark.gpu
@pytest.mark.parametrize("c", _UNCHANGED, ids=lambda c: c["name"])
def test_requesting_input_grads_changes_nothing_else(c):
    """Outputs, dL/dx, dL/dv and every parameter gradient are bitwise those of a run without the new gradients."""
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    runs = []
    for want in (False, True):
        m = make_model(c, d)
        got = _cuda_run(c, m, inp, G, want=want)
        got["params"] = {k: q.grad.detach().cpu().clone() for k, q in m.named_parameters() if q.grad is not None}
        runs.append(got)
    a, b = runs
    for k in ("x", "v", "h", "gx", "gv"):
        assert torch.equal(a[k], b[k]), k
    assert a["params"].keys() == b["params"].keys()
    for k in a["params"]:
        assert torch.equal(a["params"][k], b["params"][k]), k


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


_EGRAD_NAME = re.compile(r"k_edge_bwd_sel<(true|false), true>|k_edge_bwd<true>")
_NEW_KERNELS = ("k_sum_slices", "k_embed_input_grad", "k_loc_mean_grad")


@pytest.mark.gpu
def test_a_step_without_input_grads_launches_nothing_new():
    c = egno("egno_cfg3_full", 101, B=256, N=20, T=10, L=4)
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    m = make_model(c, d)
    lib = nb.load_library()
    counts = {}
    for want in (False, True):
        _cuda_run(c, m, inp, G, want=want)      # warm-up
        torch.cuda.synchronize()
        n0 = lib.nb_launch_count()
        _cuda_run(c, m, inp, G, want=want)
        counts[want] = lib.nb_launch_count() - n0
        names = _kernel_names(lambda: _cuda_run(c, m, inp, G, want=want))
        egrad = sorted(n for n in names if _EGRAD_NAME.search(n))
        new = sorted(n for n in names if any(k in n for k in _NEW_KERNELS))
        print(f"input grads {want}: {counts[want]} launches; EGRAD kernels {egrad}; new kernels {new}")
        assert any("k_edge_bwd_sel<false, false>" in n for n in names) != want
        if want:
            assert egrad and len(new) == len(_NEW_KERNELS)
        else:
            assert not egrad and not new
    # forward + backward launch what they launched before (62; bench.py's 65 per step add the loss and the optimizer);
    # the input gradients add exactly: sum over T, the projection, the edge-slice sum and one loc_mean kernel per layer
    assert counts[False] == 62, counts
    assert counts[True] - counts[False] == 3 + c["L"], counts


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["egno", "segno"])
def test_unrolled_training_through_two_calls_matches_float64(model):
    """A loss on the second of two chained calls, with O.egno_features / O.segno_features in between: parameter
    gradients (summed over both calls) and dL/d(initial x, v) match the same chain in float64."""
    d = _dev()
    c = egno("chain", 111, B=4, N=5, T=4, L=2) if model == "egno" else segno("chain", 112, B=4, N=5, T=4)
    B, N = c["B"], c["N"]
    m = make_model(c, d)
    w = weights_of(m)
    row, col = synth.canonical_edges(B, N)
    s = synth.sample_state("charged" if model == "egno" else "gravity", B, N, c["seed"])
    q = s["charges"]
    t_out = torch.arange(1, c["T"] + 1)[None].repeat(B, 1)
    gen = torch.Generator().manual_seed(5)
    Gx = torch.randn(B * N * (c["T"] if model == "egno" else 1), 3, generator=gen)
    Gv = torch.randn(Gx.shape, generator=gen)

    def chain(run_call, x0, v0, qq, r, cc):   # the second call starts from the first one's last predicted frame
        xo, vo = run_call(x0, v0, qq, r, cc)
        k = B * N
        return run_call(xo[-k:], vo[-k:], qq, r, cc)

    def run_egno_cuda(x, v, qq, r, cc):
        _, _, ea, nodes, lm = O.egno_features(x.view(B, N, 3), v.view(B, N, 3), qq, r, cc)
        xo, vo, _ = m(x, nodes, [r, cc], ea, v=v, loc_mean=lm, timesteps_out=t_out.to(d))
        return xo, vo

    def run_segno_cuda(x, v, qq, r, cc):
        his, _, _, ea = O.segno_features(x.view(B, N, 3), v.view(B, N, 3), qq, r, cc)
        xo, _, vo = m(his.contiguous(), x, [r, cc], v, ea.contiguous(), T=c["T"])
        return xo, vo

    p = {k: t.double().requires_grad_(True) for k, t in w.items()}

    def run_egno_ref(x, v, qq, r, cc):
        _, _, ea, nodes, lm = O.egno_features(x.view(B, N, 3), v.view(B, N, 3), qq, r, cc)
        xo, vo, _ = O.egno_forward(p, x, nodes, r, cc, ea, v, lm, t_out, n_layers=c["L"], num_timesteps=c["T"],
                                   time_emb_dim=c["time_emb_dim"], use_time_conv=True)
        return xo, vo

    def run_segno_ref(x, v, qq, r, cc):
        his, _, _, ea = O.segno_features(x.view(B, N, 3), v.view(B, N, 3), qq, r, cc)
        xo, _, vo = O.segno_forward(p, his, x, r, cc, v, ea, c["T"], recurrent=c["recurrent"],
                                    coords_weight=c["coords_weight"])
        return xo, vo

    x0 = s["loc"].reshape(-1, 3).to(d).requires_grad_(True)
    v0 = s["vel"].reshape(-1, 3).to(d).requires_grad_(True)
    xo, vo = chain(run_egno_cuda if model == "egno" else run_segno_cuda, x0, v0, q.to(d), row.to(d), col.to(d))
    ((xo * Gx.to(d)).sum() + (vo * Gv.to(d)).sum()).backward()
    xr = s["loc"].reshape(-1, 3).double().requires_grad_(True)
    vr = s["vel"].reshape(-1, 3).double().requires_grad_(True)
    xor, vor = chain(run_egno_ref if model == "egno" else run_segno_ref, xr, vr, q.double(), row, col)
    ((xor * Gx.double()).sum() + (vor * Gv.double()).sum()).backward()
    errs = dict(x=rel_err(xo.detach().cpu(), xor.detach()), gx=rel_err(x0.grad.cpu(), xr.grad),
                gv=rel_err(v0.grad.cpu(), vr.grad))
    for k, q_ in m.named_parameters():
        if p[k].grad is None:
            assert q_.grad is None or not bool(q_.grad.any()), k
            continue
        errs[k] = rel_err(q_.grad.cpu(), p[k].grad)
    worst = max(errs.items(), key=lambda kv: kv[1])
    print(f"{model} two-call chain: worst rel err {worst[0]} {worst[1]:.1e}")
    for k, e in errs.items():
        assert e < TOL_GRAD, (k, e)


# ---- guard bands around the raw entry points
def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,T,L", [(3, 20, 10, 2), (2, 29, 4, 2)])
def test_egno_backward_ex_never_writes_outside_its_buffers(B, N, T, L):
    from tests.test_gpu_guards import SENT, Arena
    d = _dev()
    lib = nb.load_library()
    row, col = synth.canonical_edges(B, N)
    s = synth.sample_state("charged", B, N, seed=7)
    x, nodes, ea, v, lm = [t.to(d).contiguous() for t in synth.egno_features(s["loc"], s["vel"], s["charges"], row, col)]
    cfg = _cabi.NbEgnoConfig(B, N, T, L, 2, 2, 2, 32, 1, 1)
    npar = lib.nb_egno_param_count(ctypes.byref(cfg))
    params = (0.1 * torch.randn(npar, generator=torch.Generator().manual_seed(1))).to(d)
    ts = torch.arange(1, T + 1, device=d)[None].repeat(B, 1).contiguous()
    Nn, n0, E0 = T * B * N, B * N, B * N * (N - 1)
    st = ctypes.c_void_p(torch.cuda.current_stream(d).cuda_stream)
    A = Arena(dict(x_out=Nn * 3, v_out=Nn * 3, h_out=Nn * 64, saved=lib.nb_egno_saved_floats(ctypes.byref(cfg)),
                   ws_f=lib.nb_egno_workspace_floats(ctypes.byref(cfg), 2), ws_b=lib.nb_egno_workspace_floats(ctypes.byref(cfg), 1),
                   iws=lib.nb_egno_input_grad_workspace_floats(ctypes.byref(cfg)), grad=npar, gx_in=n0 * 3, gv_in=n0 * 3,
                   g_nodes=n0 * 2, g_ef=E0 * 2, g_lm=n0 * 3), d)
    rc = lib.nb_egno_forward(ctypes.byref(cfg), _p(params), _p(x), _p(nodes), _p(ea), _p(v), _p(lm), _p(ts), None, A.ptr("x_out"),
                             A.ptr("v_out"), A.ptr("h_out"), A.ptr("saved"), A.ptr("ws_f"), st)
    assert rc == 0, lib.nb_last_error()
    g = torch.Generator().manual_seed(2)
    Gx, Gv, Gh = [torch.randn(Nn, k, generator=g).to(d) for k in (3, 3, 64)]
    rc = lib.nb_egno_backward_ex(ctypes.byref(cfg), _p(params), _p(nodes), _p(ea), _p(lm), _p(ts), None, A.ptr("saved"), _p(Gx),
                                 _p(Gv), _p(Gh), A.ptr("grad"), A.ptr("gx_in"), A.ptr("gv_in"), A.ptr("g_nodes"), A.ptr("g_ef"),
                                 A.ptr("g_lm"), A.ptr("ws_b"), A.ptr("iws"), st)
    assert rc == 0, lib.nb_last_error()
    torch.cuda.synchronize()
    assert A.guards_intact()
    for k in ("grad", "gx_in", "gv_in", "g_nodes", "g_ef", "g_lm"):
        assert not bool((A.view(k) == SENT).any()), k
        assert bool(torch.isfinite(A.view(k)).all()), k


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,T", [(3, 20, 10), (2, 29, 3)])
def test_segno_backward_ex_never_writes_outside_its_buffers(B, N, T):
    from tests.test_gpu_guards import SENT, Arena
    d = _dev()
    lib = nb.load_library()
    s = synth.sample_state("gravity", B, N, seed=9)
    row, col = synth.canonical_edges(B, N)
    his, x, v, ea = [t.to(d).contiguous() for t in synth.segno_features(s["loc"], s["vel"], s["charges"], row, col)]
    cfg = _cabi.NbSegnoConfig(B, N, T, 1, 2, 1, 1.0, 0)
    npar = lib.nb_segno_param_count(ctypes.byref(cfg))
    params = (0.1 * torch.randn(npar, generator=torch.Generator().manual_seed(1))).to(d)
    Nn, E0 = B * N, B * N * (N - 1)
    st = ctypes.c_void_p(torch.cuda.current_stream(d).cuda_stream)
    A = Arena(dict(x_out=Nn * 3, h_out=Nn * 64, v_out=Nn * 3, saved=lib.nb_segno_saved_floats(ctypes.byref(cfg)),
                   ws_f=lib.nb_segno_workspace_floats(ctypes.byref(cfg), 2), ws_b=lib.nb_segno_workspace_floats(ctypes.byref(cfg), 1),
                   iws=lib.nb_segno_input_grad_workspace_floats(ctypes.byref(cfg)), grad=npar, gx_in=Nn * 3, gv_in=Nn * 3,
                   g_his=Nn, g_ea=E0 * 2), d)
    rc = lib.nb_segno_forward(ctypes.byref(cfg), _p(params), _p(his), _p(x), _p(v), _p(ea), A.ptr("x_out"), A.ptr("h_out"),
                              A.ptr("v_out"), A.ptr("saved"), A.ptr("ws_f"), st)
    assert rc == 0, lib.nb_last_error()
    g = torch.Generator().manual_seed(2)
    Gx, Gh, Gv = [torch.randn(Nn, k, generator=g).to(d) for k in (3, 64, 3)]
    rc = lib.nb_segno_backward_ex(ctypes.byref(cfg), _p(params), _p(his), _p(ea), A.ptr("saved"), _p(Gx), _p(Gh), _p(Gv),
                                  A.ptr("grad"), A.ptr("gx_in"), A.ptr("gv_in"), None, A.ptr("g_his"), A.ptr("g_ea"),
                                  A.ptr("ws_b"), A.ptr("iws"), st)
    assert rc == 0, lib.nb_last_error()
    torch.cuda.synchronize()
    assert A.guards_intact()
    for k in ("grad", "gx_in", "gv_in", "g_his", "g_ea"):
        assert not bool((A.view(k) == SENT).any()), k
        assert bool(torch.isfinite(A.view(k)).all()), k


@pytest.mark.gpu
@pytest.mark.parametrize("c", [egno("egno_det_N20", 121, B=16, N=20, T=10, L=2), egno("egno_det_N29", 122, B=3, N=29, T=4, L=2),
                               segno("segno_det_N20", 123, B=16, N=20, T=6)], ids=lambda c: c["name"])
def test_input_grads_are_bitwise_deterministic(c):
    d = _dev()
    inp = make_inputs(c)
    G = cotangents(c)
    a, b = (_cuda_run(c, make_model(c, d), inp, G) for _ in range(2))
    for k in NEW[c["model"]]:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
def test_edge_grads_under_the_tc_cross_check_kernels_raise():
    c = egno("egno_impl1", 131, B=3, N=5, T=4, L=1)
    d = _dev()
    lib = nb.load_library()
    inp = make_inputs(c)
    G = cotangents(c)
    m = make_model(c, d)
    assert lib.nb_set_edge_impl(1) == 0
    try:
        with pytest.raises(RuntimeError, match="nb_set_edge_impl\\(1\\)"):
            _cuda_run(c, m, inp, G)
    finally:
        lib.nb_set_edge_impl(2)
    assert lib.nb_get_edge_impl() == 2
