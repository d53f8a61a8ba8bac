"""The three-tiles-in-flight edge forward (k_edge_fwd_sel3) against the two-CTA-per-SM kernel it replaces for units of
at least three tiles: M and Fsum bitwise equal across the shapes it takes, a whole EGNO training step bitwise equal
with it on and off, and the launch selection (N = 20 takes it, N = 5 and N = 100 do not)."""
import ctypes
import re

import pytest
import torch

import no_node_comparison_b200 as nb
from no_node_comparison_b200 import synth

pytestmark = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    return torch.device("cuda:0")


def _edge_forward(lib, n_gt, B, N, nef, clamp, t):
    d = dev()
    M = torch.full((n_gt * N, 64), float("nan"), device=d)
    F = torch.full((n_gt * N, 3), float("nan"), device=d)
    ptr = lambda x: ctypes.c_void_p(x.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.nb_egcl_edge_forward(n_gt, B, N, nef, clamp, ptr(t["x"]), ptr(t["P"]), ptr(t["Q"]), ptr(t["ef"]), ptr(t["w1"]),
                                  1 + nef, 0, 1, ptr(t["W2"]), ptr(t["b2"]), ptr(t["W3"]), ptr(t["b3"]), ptr(t["w4"]),
                                  ptr(t["b4"]), ptr(M), ptr(F), st)
    assert rc == 0, lib.nb_last_error()
    torch.cuda.synchronize()
    return M.cpu(), F.cpu()


@pytest.mark.parametrize("clamp", [0, 1])
@pytest.mark.parametrize("nef", [0, 2, 4])
@pytest.mark.parametrize("N", [17, 20, 21, 27])
def test_three_tile_forward_is_bitwise_equal(N, nef, clamp):
    """3, 3, 4 and 6 tiles per unit (the last one partial at every N); 1024 graph-instances over B = 256 edge-feature
    graphs, so every CTA walks several units and both node-tile buffers; with the clamp on, positions are scaled so
    that many edge forces saturate it."""
    lib = nb.load_library()
    d = dev()
    B, n_gt = 256, 1024
    gen = torch.Generator().manual_seed(N * 100 + nef * 10 + clamp)
    nn_ = n_gt * N
    t = dict(x=torch.randn(nn_, 3, generator=gen) * (20.0 if clamp else 1.0),
             P=torch.randn(nn_, 64, generator=gen) * 0.5, Q=torch.randn(nn_, 64, generator=gen) * 0.5,
             ef=torch.randn(max(1, B * N * (N - 1) * nef), generator=gen),
             w1=torch.randn(64, 1 + nef, generator=gen) * 0.3,
             W2=torch.randn(64, 64, generator=gen) * 0.15, W3=torch.randn(64, 64, generator=gen) * 0.15,
             b2=torch.randn(64, generator=gen) * 0.1, b3=torch.randn(64, generator=gen) * 0.1,
             w4=torch.randn(64, generator=gen) * 0.5, b4=torch.randn(1, generator=gen))
    t = {k: v.to(d).contiguous() for k, v in t.items()}
    assert lib.nb_get_edge_fwd3() == 1
    M3, F3 = _edge_forward(lib, n_gt, B, N, nef, clamp, t)
    assert lib.nb_set_edge_fwd3(0) == 0
    try:
        M2, F2 = _edge_forward(lib, n_gt, B, N, nef, clamp, t)
    finally:
        lib.nb_set_edge_fwd3(1)
    assert torch.isfinite(M3).all() and torch.isfinite(F3).all()
    assert torch.equal(M3, M2)
    assert torch.equal(F3, F2)


def _egno_step(B, N, T, seed=3):
    """Outputs and every gradient of one EGNO training step at (B, N, T), 4 layers."""
    d = dev()
    torch.manual_seed(1)
    m = nb.EGNO(n_layers=4, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T, device=d)
    row, col = synth.canonical_edges(B, N)
    s = synth.sample_state("charged", B, N, seed=seed)
    edges = [row.to(d), col.to(d)]
    x, nodes, ea, v, lm = synth.egno_features(s["loc"].to(d), s["vel"].to(d), s["charges"].to(d), edges[0], edges[1])
    x = x.clone().requires_grad_(True)
    v = v.clone().requires_grad_(True)
    t_out = torch.arange(1, T + 1, device=d)[None].repeat(B, 1)
    xo, vo, ho = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
    g = torch.Generator(device=d).manual_seed(7)
    (xo * torch.randn(xo.shape, generator=g, device=d)).sum().add((ho * ho).mean()).add((vo * vo).sum()).backward()
    torch.cuda.synchronize()
    return [xo.detach().cpu(), vo.detach().cpu(), ho.detach().cpu(), x.grad.cpu(), v.grad.cpu()] + \
        [p.grad.detach().cpu().clone() for p in m.parameters()]


def test_egno_training_step_is_bitwise_equal():
    """The benchmark's EGNO configuration (B = 256, N = 20, T = 10, 4 layers): outputs, input gradients and every
    parameter gradient are bitwise equal with the three-tile forward on and off."""
    lib = nb.load_library()
    on = _egno_step(256, 20, 10)
    assert lib.nb_set_edge_fwd3(0) == 0
    try:
        off = _egno_step(256, 20, 10)
    finally:
        lib.nb_set_edge_fwd3(1)
    assert len(on) == len(off) > 5
    for a, b in zip(on, off):
        assert torch.equal(a, b)


def _edge_fwd_kernels(B, N, T):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _egno_step(B, N, T)
    return {re.search(r"k_edge_fwd\w*", e.name).group(0) for e in prof.events() if "k_edge_fwd" in e.name}


def test_launch_selection_follows_unit_geometry():
    """N = 20 (three tiles per graph-instance) runs k_edge_fwd_sel3; N = 5 (packed units of one tile) and N = 100 (the
    blocked walk) run k_edge_fwd_sel."""
    assert _edge_fwd_kernels(256, 20, 10) == {"k_edge_fwd_sel3"}
    assert _edge_fwd_kernels(64, 5, 8) == {"k_edge_fwd_sel"}
    assert _edge_fwd_kernels(2, 100, 4) == {"k_edge_fwd_sel"}
