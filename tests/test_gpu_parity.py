"""Parity of the CUDA path (through the drop-in modules -> C ABI -> sm_100a kernels) against the golden
vectors of the reference and against the oracle; plus size-independent properties at BASELINE sizes.

Tolerances (fp32 everywhere; BASELINE.json: predicted positions rel. err <= 1e-4):
  outputs   : max|a-b| / max|b| <= 1e-4   (observed ~1e-6 .. 1e-5: summation order + split-bf16 operands)
  gradients : <= 1e-3                       (observed ~1e-5)
EGNO parameter gradients are held to 1e-3 (scale-relative) on EVERY entry of every tensor except TimeConv's own weights,
where a counted budget applies (helpers.param_grads_within_kink_budget: at most 1e-4 of the layer's activations may take
the other LeakyReLU slope, each moving at most 64 gradient entries, none by more than 2e-2): TimeConv applies LeakyReLU to the
spectral convolution of h (layer_no.py:125-126), and an element whose pre-activation is within rounding distance of the
kink takes the other slope under ANY change of summation order or operand rounding upstream (the reference itself does
so between CPU and GPU, or with TF32).  One flipped element moves one column of that layer's weight gradient by
O(1/(B*N)) of its scale (observed: 36 of 16 384 entries by 0.6 % in the (8,20,10,4) case) and nothing else visibly.
The fp32 SIMT variants of the kernels are held to the strict max-norm bound in test_kernel_variants_agree_on_golden_case.
"""
import math

import pytest
import torch

import no_node_comparison_b200 as nb
from no_node_comparison_b200 import synth
from oracle import nbody_oracle as O
from tests.helpers import (EGNO_CASES, EGNO_MULTI_CASES, SEGNO_CASES, SEGNO_MULTI_CASES, load_case, rel_err, rel_l2,
                           param_grads_within_kink_budget,
                           egno_inputs_from_case, egno_multi_inputs_from_case, segno_inputs_from_case,
                           segno_multi_inputs_from_case)

pytestmark = pytest.mark.gpu
TOL_OUT = 1e-4
TOL_GRAD = 1e-3


def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    return torch.device("cuda:0")


def make_egno(c, w=None, seed=1):
    torch.manual_seed(seed)
    m = nb.EGNO(n_layers=c["L"], in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=c["modes"],
                num_timesteps=c["T"], device=dev())
    if w is not None:
        m.load_state_dict(w)
    return m


def run_egno(m, c, requires_grad=True):
    d = dev()
    x = c["x"].to(d).requires_grad_(requires_grad)
    v = c["v"].to(d).requires_grad_(requires_grad)
    out = m(x, c["nodes"].to(d), [c["row"].to(d), c["col"].to(d)], c["edge_attr"].to(d), v=v,
            loc_mean=c["loc_mean"].to(d), timesteps_out=c["t_out"].to(d))
    return x, v, out


@pytest.mark.parametrize("name", EGNO_CASES)
def test_egno_matches_reference_golden(name):
    dd, w, g = load_case(name)
    c = egno_inputs_from_case(dd)
    m = make_egno(c, w)
    x, v, (xo, vo, ho) = run_egno(m, c)
    assert rel_err(xo.cpu(), torch.tensor(dd["x_out"])) < TOL_OUT
    assert rel_err(vo.cpu(), torch.tensor(dd["v_out"])) < TOL_OUT
    assert rel_err(ho.cpu(), torch.tensor(dd["h_out"])) < TOL_OUT
    d = dev()
    loss = (xo * torch.tensor(dd["Gx"], device=d)).sum() + (vo * torch.tensor(dd["Gv"], device=d)).sum() + \
        (ho * torch.tensor(dd["Gh"], device=d)).sum()
    loss.backward()
    assert rel_err(x.grad.cpu(), torch.tensor(dd["gx_in"])) < TOL_GRAD
    assert rel_err(v.grad.cpu(), torch.tensor(dd["gv_in"])) < TOL_GRAD
    for k, p in m.named_parameters():
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(g[k])
        assert rel_err(got, g[k]) < TOL_GRAD, k


@pytest.mark.parametrize("name", EGNO_MULTI_CASES)
def test_egno_multi_input_matches_reference_golden(name):
    """num_inputs > 1 (several input frames, a second time embedding, per-frame edge features) and per-trajectory output
    times (varDT), the PRO half of the reference's sweep (_schedule.yaml:38-68): golden vectors of the real reference."""
    dd, w, g = load_case(name)
    c = egno_multi_inputs_from_case(dd)
    d = dev()
    torch.manual_seed(1)
    m = nb.EGNO(n_layers=c["L"], in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=c["modes"],
                num_timesteps=c["T"], num_inputs=c["num_inputs"], device=d)
    m.load_state_dict(w)
    x = c["x"].to(d).requires_grad_(True)
    v = c["v"].to(d).requires_grad_(True)
    xo, vo, ho = m(x, c["nodes"].to(d), [c["row"].to(d), c["col"].to(d)], c["edge_attr"].to(d), v=v,
                   loc_mean=c["loc_mean"].to(d), timesteps_in=c["t_in"].to(d), timesteps_out=c["t_out"].to(d))
    assert rel_err(xo.cpu(), torch.tensor(dd["x_out"])) < TOL_OUT
    assert rel_err(vo.cpu(), torch.tensor(dd["v_out"])) < TOL_OUT
    assert rel_err(ho.cpu(), torch.tensor(dd["h_out"])) < TOL_OUT
    loss = (xo * torch.tensor(dd["Gx"], device=d)).sum() + (vo * torch.tensor(dd["Gv"], device=d)).sum() + \
        (ho * torch.tensor(dd["Gh"], device=d)).sum()
    loss.backward()
    assert x.grad.shape == x.shape and v.grad.shape == v.shape
    assert rel_err(x.grad.cpu(), torch.tensor(dd["gx_in"])) < TOL_GRAD
    assert rel_err(v.grad.cpu(), torch.tensor(dd["gv_in"])) < TOL_GRAD
    for k, p in m.named_parameters():
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(g[k])
        assert rel_err(got, g[k]) < TOL_GRAD, k


@pytest.mark.parametrize("name", SEGNO_CASES)
def test_segno_matches_reference_golden(name):
    dd, w, g = load_case(name)
    c = segno_inputs_from_case(dd)
    d = dev()
    m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True)
    m.load_state_dict(w)
    x = c["x"].to(d).requires_grad_(True)
    v = c["v"].to(d).requires_grad_(True)
    # edge index left on the host, as SEGNO/train_nbody.py:76-78 does
    xo, ho, vo = m(c["his"].to(d), x, [c["row"], c["col"]], v, c["edge_attr"].to(d), T=c["T"])
    assert m.n_layers == c["T"] and m.module.n_layers == c["T"]          # model.py:96-97
    assert rel_err(xo.cpu(), torch.tensor(dd["x_out"])) < TOL_OUT
    assert rel_err(vo.cpu(), torch.tensor(dd["v_out"])) < TOL_OUT
    assert rel_err(ho.cpu(), torch.tensor(dd["h_out"])) < TOL_OUT
    loss = (xo * torch.tensor(dd["Gx"], device=d)).sum() + (vo * torch.tensor(dd["Gv"], device=d)).sum() + \
        (ho * torch.tensor(dd["Gh"], device=d)).sum()
    loss.backward()
    assert rel_err(x.grad.cpu(), torch.tensor(dd["gx_in"])) < TOL_GRAD
    assert rel_err(v.grad.cpu(), torch.tensor(dd["gv_in"])) < TOL_GRAD
    for k, p in m.named_parameters():
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(g[k])
        assert rel_err(got, g[k]) < TOL_GRAD, k
    assert m.module.coord_mlp_vel[0].weight.grad is None or float(m.module.coord_mlp_vel[0].weight.grad.abs().max()) == 0


def _egno_case(B, N, T, L=2, modes=2, seed=0, kind="charged"):
    s = synth.sample_state(kind, B, N, seed)
    row, col = synth.canonical_edges(B, N)
    x, nodes, ea, v, lm = synth.egno_features(s["loc"], s["vel"], s["charges"], row, col)
    return dict(n=N, B=B, T=T, L=L, modes=modes, row=row, col=col, x=x, v=v, edge_attr=ea, nodes=nodes, loc_mean=lm,
                t_out=torch.arange(1, T + 1)[None].repeat(B, 1))


@pytest.mark.parametrize("B,N,T,L", [(8, 20, 10, 4), (1, 100, 3, 1), (5, 2, 4, 2), (3, 37, 5, 1), (13, 5, 8, 2)])
def test_egno_vs_oracle_various_shapes(B, N, T, L):
    c = _egno_case(B, N, T, L=L, seed=B + N)
    m = make_egno(c)
    w = {k: t.detach().cpu().clone() for k, t in m.state_dict().items()}
    x, v, (xo, vo, ho) = run_egno(m, c)
    gen = torch.Generator().manual_seed(3)
    Gx, Gh = torch.randn(xo.shape, generator=gen), torch.randn(ho.shape, generator=gen) * 0.05
    ((xo * Gx.to(dev())).sum() + (ho * Gh.to(dev())).sum()).backward()
    p = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    xr = c["x"].clone().requires_grad_(True)
    xo_r, vo_r, ho_r = O.egno_forward(p, xr, c["nodes"], c["row"], c["col"], c["edge_attr"], c["v"], c["loc_mean"],
                                      c["t_out"], n_layers=L, num_timesteps=T)
    ((xo_r * Gx).sum() + (ho_r * Gh).sum()).backward()
    assert rel_err(xo.cpu(), xo_r.detach()) < TOL_OUT
    assert rel_err(vo.cpu(), vo_r.detach()) < TOL_OUT
    assert rel_err(ho.cpu(), ho_r.detach()) < TOL_OUT
    assert rel_err(x.grad.cpu(), xr.grad) < TOL_GRAD
    param_grads_within_kink_budget(m, p, n_rows=T * B * N, tol=TOL_GRAD)


@pytest.mark.parametrize("B,N,T", [(16, 20, 10), (2, 100, 2), (9, 3, 5), (3, 27, 4), (2, 28, 3)])   # 27: largest fused unit; 28: blocked walk
def test_segno_vs_oracle_various_shapes(B, N, T):
    d = dev()
    s = synth.sample_state("gravity", B, N, seed=B)
    row, col = synth.canonical_edges(B, N)
    his, x0, v0, ea = synth.segno_features(s["loc"], s["vel"], s["charges"], row, col)
    torch.manual_seed(2)
    m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True)
    with torch.no_grad():
        m.module.coord_mlp[2].weight.mul_(200.0)     # make the coordinate path numerically visible
    w = {k: t.detach().cpu().clone() for k, t in m.state_dict().items()}
    x = x0.to(d).requires_grad_(True)
    xo, ho, vo = m(his.to(d), x, torch.stack([row, col]).to(d), v0.to(d), ea.to(d), T=T)
    gen = torch.Generator().manual_seed(4)
    Gx, Gv = torch.randn(xo.shape, generator=gen), torch.randn(vo.shape, generator=gen)
    ((xo * Gx.to(d)).sum() + (vo * Gv.to(d)).sum()).backward()
    p = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    xr = x0.clone().requires_grad_(True)
    xo_r, ho_r, vo_r = O.segno_forward(p, his, xr, row, col, v0, ea, T)
    ((xo_r * Gx).sum() + (vo_r * Gv).sum()).backward()
    assert rel_err(xo.cpu(), xo_r.detach()) < TOL_OUT
    assert rel_err(vo.cpu(), vo_r.detach()) < TOL_OUT
    assert rel_err(ho.cpu(), ho_r.detach()) < TOL_OUT
    assert rel_err(x.grad.cpu(), xr.grad) < TOL_GRAD
    for k, q in m.named_parameters():
        ref = p[k].grad if p[k].grad is not None else torch.zeros_like(p[k])
        got = q.grad.cpu() if q.grad is not None else torch.zeros_like(ref)
        assert rel_err(got, ref) < TOL_GRAD, k


def _rotation(seed=0):
    g = torch.Generator().manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
    if torch.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q


def test_egno_full_size_properties():
    """BASELINE config 3 size (N=20, T=10, L=4, B=256): E(3) equivariance, batch independence,
    data-parallel equivalence of gradients, bitwise determinism, no_grad == grad forward."""
    d = dev()
    B, N, T = 256, 20, 10
    c = _egno_case(B, N, T, L=4, seed=11)
    m = make_egno(c)
    x, v, (xo, vo, ho) = run_egno(m, c)
    loss = (xo ** 2).mean() + (ho ** 2).mean()
    loss.backward()
    g_full = torch.cat([p.grad.reshape(-1) for p in m.parameters()]).clone()
    # determinism: same inputs -> bit-identical outputs and gradients (no atomics anywhere)
    m.zero_grad()
    x2, v2, (xo2, vo2, ho2) = run_egno(m, c)
    ((xo2 ** 2).mean() + (ho2 ** 2).mean()).backward()
    assert torch.equal(xo, xo2) and torch.equal(ho, ho2)
    assert torch.equal(g_full, torch.cat([p.grad.reshape(-1) for p in m.parameters()]))
    # inference path (nothing saved) gives the same numbers
    with torch.no_grad():
        _, _, (xo3, vo3, ho3) = run_egno(m, c, requires_grad=False)
    assert torch.equal(xo, xo3) and torch.equal(vo, vo3) and torch.equal(ho, ho3)
    # E(3): rotate + translate positions, rotate velocities -> outputs rotate/translate, h invariant
    R, t = _rotation(1), torch.tensor([0.3, -1.2, 0.7])
    s = synth.sample_state("charged", B, N, 11)
    row, col = c["row"], c["col"]
    xr, nodes_r, ea_r, vr, lm_r = synth.egno_features(s["loc"] @ R.T + t, s["vel"] @ R.T, s["charges"], row, col)
    cr = dict(c, x=xr, v=vr, nodes=nodes_r, edge_attr=ea_r, loc_mean=lm_r)
    with torch.no_grad():
        _, _, (xo_r, vo_r, ho_r) = run_egno(m, cr, requires_grad=False)
    Rd, td = R.to(d), t.to(d)
    assert rel_err(xo_r, xo.detach() @ Rd.T + td) < 5e-5
    assert rel_err(vo_r, vo.detach() @ Rd.T) < 5e-5
    assert rel_err(ho_r, ho.detach()) < 5e-5
    # batch independence + DP equivalence: two half batches reproduce outputs; mean of their grads == full grads
    halves, g_halves = [], []
    for lo in (0, B // 2):
        sl = {k: s[k][lo:lo + B // 2] for k in s}
        rr, cc = synth.canonical_edges(B // 2, N)
        xh, nh, eh, vh, lmh = synth.egno_features(sl["loc"], sl["vel"], sl["charges"], rr, cc)
        ch = dict(c, B=B // 2, row=rr, col=cc, x=xh, v=vh, nodes=nh, edge_attr=eh, loc_mean=lmh, t_out=c["t_out"][:B // 2])
        m.zero_grad()
        _, _, (xh_o, vh_o, hh_o) = run_egno(m, ch)
        ((xh_o ** 2).mean() + (hh_o ** 2).mean()).backward()
        halves.append(xh_o.detach().view(T, B // 2 * N, 3))
        g_halves.append(torch.cat([p.grad.reshape(-1) for p in m.parameters()]).clone())
    xo_cat = torch.cat(halves, dim=1).reshape(-1, 3)
    assert rel_err(xo_cat, xo.detach()) < 1e-6
    assert rel_err(0.5 * (g_halves[0] + g_halves[1]), g_full) < 1e-4


def test_segno_full_size_equivariance_and_rollout_energy():
    """BASELINE config 4 size (gravity, N=20, T=10, B=256): E(3) equivariance and a short GPU-resident
    rollout whose energies are finite and computed identically to the oracle's energy function."""
    d = dev()
    B, N, T = 256, 20, 10
    s = synth.sample_state("gravity", B, N, seed=5)
    row, col = synth.canonical_edges(B, N)
    torch.manual_seed(1)
    m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True)
    with torch.no_grad():
        m.module.coord_mlp[2].weight.mul_(100.0)
    edges = [row.to(d), col.to(d)]

    def run(loc, vel):
        his, x, v, ea = synth.segno_features(loc, vel, s["charges"], row, col)
        with torch.no_grad():
            return m(his.to(d), x.to(d), edges, v.to(d), ea.to(d), T=T)

    xo, ho, vo = run(s["loc"], s["vel"])
    R, t = _rotation(2), torch.tensor([1.0, 2.0, -0.5])
    xo_r, ho_r, vo_r = run(s["loc"] @ R.T + t, s["vel"] @ R.T)
    Rd, td = R.to(d), t.to(d)
    assert rel_err(xo_r, xo @ Rd.T + td) < 5e-5
    assert rel_err(vo_r, vo @ Rd.T) < 5e-5
    assert rel_err(ho_r, ho) < 5e-5
    # 3-call rollout (train_nbody.py:200-236): features recomputed from the prediction each call
    loc, vel = s["loc"], s["vel"]
    for _ in range(3):
        xo, ho, vo = run(loc, vel)
        loc, vel = xo.cpu().view(B, N, 3), vo.cpu().view(B, N, 3)
        e = O.energy_gravity(loc, vel, s["charges"])
        assert torch.isfinite(e).all()


def test_training_steps_follow_the_oracle():
    """Three Adam steps (lr from model_confs.yaml:16) on the CUDA path track the oracle's loss curve."""
    d = dev()
    c = _egno_case(16, 5, 8, L=4, seed=21)
    target = torch.randn(8 * 16 * 5, 3, generator=torch.Generator().manual_seed(9)) * 0.1 + c["x"].repeat(8, 1)
    m = make_egno(c)
    w = {k: t.detach().cpu().clone() for k, t in m.state_dict().items()}
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        _, _, (xo, vo, ho) = run_egno(m, c, requires_grad=False)
        loss = ((xo - target.to(d)) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    p = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    opt_r = torch.optim.Adam(list(p.values()), lr=1e-3)
    ref_losses = []
    for _ in range(3):
        opt_r.zero_grad()
        xo_r, _, _ = O.egno_forward(p, c["x"], c["nodes"], c["row"], c["col"], c["edge_attr"], c["v"], c["loc_mean"],
                                    c["t_out"], n_layers=4, num_timesteps=8)
        loss = ((xo_r - target) ** 2).mean()
        loss.backward()
        opt_r.step()
        ref_losses.append(loss.item())
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 1e-4 * abs(b) + 1e-7, (losses, ref_losses)


def test_non_canonical_edges_raise_on_device():
    d = dev()
    c = _egno_case(4, 5, 8, L=1)
    m = make_egno(c)
    col = c["col"].clone()
    col[0], col[1] = c["col"][1], c["col"][0]
    with pytest.raises(ValueError, match="canonical"):
        m(c["x"].to(d), c["nodes"].to(d), [c["row"].to(d), col.to(d)], c["edge_attr"].to(d), v=c["v"].to(d),
          loc_mean=c["loc_mean"].to(d), timesteps_out=c["t_out"].to(d))
    with pytest.raises(ValueError):
        m(c["x"].to(d), c["nodes"].to(d), [c["row"].to(d), c["col"].to(d)], c["edge_attr"].to(d), v=c["v"].to(d),
          loc_mean=c["loc_mean"].to(d), timesteps_out=c["t_out"][:, :4].to(d))


@pytest.mark.parametrize("impl", [2, 0])
def test_edge_tile_building_block_vs_oracle(impl):
    """nb_egcl_edge_forward / _backward alone (C ABI, raw pointers) against a plain edge-list evaluation, for the
    tcgen05 tiles with tensor-core gathers / scatters (impl 2, the default; split-bf16 operands: ~1e-5) and the fp32
    SIMT tiles (impl 0: ~1e-6)."""
    import ctypes
    d = dev()
    lib = nb.load_library()
    assert lib.nb_set_edge_impl(impl) == 0
    try:
        _edge_tile_check(lib, d, 5e-5 if impl >= 1 else 1e-5)
    finally:
        lib.nb_set_edge_impl(2)


def _edge_tile_check(lib, d, tol):
    import ctypes
    n_gt, B, N, nef = 12, 4, 20, 2
    gen = torch.Generator().manual_seed(0)
    nn_ = n_gt * N
    x = torch.randn(nn_, 3, generator=gen)
    P, Q = torch.randn(nn_, 64, generator=gen) * 0.5, torch.randn(nn_, 64, generator=gen) * 0.5
    ef = torch.randn(B * N * (N - 1), nef, generator=gen)
    w1 = torch.randn(64, 1 + nef, generator=gen) * 0.3
    W2, W3 = torch.randn(64, 64, generator=gen) * 0.15, torch.randn(64, 64, generator=gen) * 0.15
    b2, b3, w4, b4 = [torch.randn(n, generator=gen) * 0.1 for n in (64, 64, 64, 1)]
    gM, gF = torch.randn(nn_, 64, generator=gen), torch.randn(nn_, 3, generator=gen)
    row, col = O.canonical_edges(n_gt, N)
    eidx = (torch.arange(n_gt).repeat_interleave(N * (N - 1)) % B) * (N * (N - 1)) + torch.arange(N * (N - 1)).repeat(n_gt)
    leaves = [t.clone().requires_grad_(True) for t in (x, P, Q, w1, W2, b2, W3, b3, w4, b4)]
    xr, Pr, Qr, w1r, W2r, b2r, W3r, b3r, w4r, b4r = leaves
    rij = xr[row] - xr[col]
    r2 = (rij ** 2).sum(1, keepdim=True)
    z1 = O.silu(Pr[row] + Qr[col] + r2 * w1r[:, 0] + ef[eidx] @ w1r[:, 1:].t())
    mm = O.silu(z1 @ W2r.t() + b2r)
    cc = O.silu(mm @ W3r.t() + b3r) @ w4r[:, None] + b4r
    M_ref = O.segment_sum(mm, row, nn_)
    F_ref = O.segment_sum(rij * cc, row, nn_)
    ((M_ref * gM).sum() + (F_ref * gF).sum()).backward()
    dv = lambda t: t.detach().to(d).contiguous()
    X, Pd, Qd, EF, W1, W2d, B2, W3d, B3, W4, B4, GM, GF = map(dv, (x, P, Q, ef, w1, W2, b2, W3, b3, w4, b4, gM, gF))
    M = torch.empty(nn_, 64, device=d)
    F = torch.empty(nn_, 3, device=d)
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.nb_egcl_edge_forward(n_gt, B, N, nef, 0, ptr(X), ptr(Pd), ptr(Qd), ptr(EF), ptr(W1), 1 + nef, 0, 1,
                                  ptr(W2d), ptr(B2), ptr(W3d), ptr(B3), ptr(W4), ptr(B4), ptr(M), ptr(F), st)
    assert rc == 0, lib.nb_last_error()
    assert rel_err(M.cpu(), M_ref.detach()) < tol
    assert rel_err(F.cpu(), F_ref.detach()) < tol
    gP, gQ = torch.empty(nn_, 64, device=d), torch.empty(nn_, 64, device=d)
    gx = torch.zeros(nn_, 3, device=d)
    gw = torch.empty(2 * 4096 + 3 * 64 + 64 * (1 + nef) + 1, device=d)
    ws = torch.empty(lib.nb_egcl_edge_backward_workspace_floats(n_gt, N), device=d)
    rc = lib.nb_egcl_edge_backward(n_gt, B, N, nef, 0, ptr(X), ptr(Pd), ptr(Qd), ptr(EF), ptr(W1), 1 + nef, 0, 1,
                                   ptr(W2d), ptr(B2), ptr(W3d), ptr(B3), ptr(W4), ptr(B4), ptr(GM), ptr(GF), ptr(gP),
                                   ptr(gQ), ptr(gx), ptr(gw), ptr(ws), st)
    assert rc == 0, lib.nb_last_error()
    assert rel_err(gP.cpu(), Pr.grad) < tol
    assert rel_err(gQ.cpu(), Qr.grad) < tol
    assert rel_err(gx.cpu(), xr.grad) < tol
    gwc = gw.cpu()
    assert rel_err(gwc[:4096].view(64, 64), W2r.grad) < tol
    assert rel_err(gwc[4096:8192].view(64, 64), W3r.grad) < tol
    o = 8192
    assert rel_err(gwc[o:o + 64], b2r.grad) < tol
    assert rel_err(gwc[o + 64:o + 128], b3r.grad) < tol
    assert rel_err(gwc[o + 128:o + 192], w4r.grad) < tol
    assert rel_err(gwc[o + 192:o + 192 + 64 * (1 + nef)].view(64, 1 + nef), w1r.grad) < tol
    assert rel_err(gwc[-1:], b4r.grad) < tol


@pytest.mark.parametrize("edge_impl,node_impl", [(0, 0), (2, 0)])
def test_kernel_variants_agree_on_golden_case(edge_impl, node_impl):
    """The non-default kernel variants (fp32 SIMT edge tiles / node GEMMs) stay parity-green against the reference's
    golden vectors: they are the independent cross-checks of the default tcgen05 path (edge impl 2, node impl 1),
    which every other test in this file runs.  Any other edge impl is refused and leaves the selection as it was."""
    lib = nb.load_library()
    assert lib.nb_set_edge_impl(edge_impl) == 0 and lib.nb_set_node_impl(node_impl) == 0
    try:
        test_egno_matches_reference_golden("egno_n20_t10")
        test_segno_matches_reference_golden("segno_n5_t10")
    finally:
        lib.nb_set_edge_impl(2)
        lib.nb_set_node_impl(1)
    assert lib.nb_get_edge_impl() == 2 and lib.nb_get_node_impl() == 1
    assert lib.nb_set_edge_impl(1) != 0 and lib.nb_get_edge_impl() == 2


def test_segno_fused_forward_matches_stepwise_kernels():
    """The fused T-sub-step SEGNO forward (node state resident in shared memory, nb_segno_fused.cuh) and the backward
    whose node-level chain between two edge sweeps is one kernel (k_segno_node_bwd) against the
    one-kernel-sequence-per-sub-step path in both directions, at BASELINE.json configs[3] shape: outputs, input and
    parameter gradients; recurrent and non-recurrent node updates."""
    lib = nb.load_library()
    d = dev()
    B, N, T = 64, 20, 10
    s = synth.sample_state("gravity", B, N, seed=5)
    row, col = synth.canonical_edges(B, N)
    his, x, v, ea = synth.segno_features(s["loc"], s["vel"], s["charges"], row, col)
    for recurrent in (True, False):
        torch.manual_seed(3)
        m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=recurrent)
        out = {}
        for fused in (1, 0):
            assert lib.nb_set_segno_fused(fused) == 0
            try:
                m.zero_grad(set_to_none=True)
                xg = x.to(d).requires_grad_(True)
                vg = v.to(d).requires_grad_(True)
                n0 = lib.nb_launch_count()
                xo, ho, vo = m(his.to(d), xg, [row, col], vg, ea.to(d), T=T)
                (xo.square().sum() + 0.1 * ho.sum() + vo.square().sum()).backward()
                launches = lib.nb_launch_count() - n0
                out[fused] = [xo.detach().cpu(), ho.detach().cpu(), vo.detach().cpu(), xg.grad.cpu(), vg.grad.cpu()] + \
                    [p.grad.cpu().clone() for p in m.parameters() if p.grad is not None]
                out[fused, "launches"] = launches
            finally:
                lib.nb_set_segno_fused(1)
        assert lib.nb_get_segno_fused() == 1
        assert out[1, "launches"] < out[0, "launches"] - 4 * (T - 1)   # T - 1 chain launches replace 4 (T - 1) + the fused forward
        for a, b in zip(out[1], out[0]):
            assert rel_err(a, b) < 2e-5


@pytest.mark.parametrize("B,N,T,L", [(16, 20, 10, 4), (7, 5, 8, 2), (2, 37, 5, 1)])
def test_egno_fused_node_kernels_match_generic_launches(B, N, T, L):
    """The per-layer node kernels (nb_egno_node.cuh: node_net + node_v_net + coordinate update forward and backward,
    the first edge layer's node halves; operands chained through tensor memory) against the generic node GEMM launches
    and coordinate-update kernels they replaced (`nb_set_node_fused(0)`): outputs, input and parameter gradients, and
    the launch count (3 + 1 launches less per layer forward... 16 per 4-layer step)."""
    lib = nb.load_library()
    c = _egno_case(B, N, T, L=L, seed=31 + N)
    gen = torch.Generator().manual_seed(9)
    n = T * B * N
    Gx, Gv, Gh = torch.randn(n, 3, generator=gen).to(dev()), torch.randn(n, 3, generator=gen).to(dev()), 0.1 * torch.randn(n, 64, generator=gen).to(dev())
    out = {}
    for fused in (1, 0):
        assert lib.nb_set_node_fused(fused) == 0
        try:
            m = make_egno(c, seed=12)
            n0 = lib.nb_launch_count()
            x, v, (xo, vo, ho) = run_egno(m, c)
            ((xo * Gx).sum() + (vo * Gv).sum() + (ho * Gh).sum()).backward()
            torch.cuda.synchronize()
            out[fused, "launches"] = lib.nb_launch_count() - n0
            out[fused] = [xo.detach().cpu(), vo.detach().cpu(), ho.detach().cpu(), x.grad.cpu(), v.grad.cpu()] + \
                [p.grad.cpu().clone() for p in m.parameters()]
        finally:
            lib.nb_set_node_fused(1)
    assert lib.nb_get_node_fused() == 1
    assert out[1, "launches"] == out[0, "launches"] - 4 * L      # 2 launches less per layer in each direction
    for a, b in zip(out[1][:5], out[0][:5]):
        assert rel_err(a, b) < 2e-5
    for a, b in zip(out[1][5:], out[0][5:]):
        assert rel_err(a, b) < 1e-3      # parameter gradients: LeakyReLU-kink flips under any rounding change (see the header)


def test_cuda_graph_training_step_matches_eager():
    """GraphedStep (forward + loss + backward + Adam captured in one CUDA graph) follows the eager step bit for bit:
    the C ABI is enqueue-only and allocation-free, so capture must not change any result."""
    d = dev()
    c = _egno_case(16, 20, 10, L=2, seed=9)
    tgt = (c["x"].repeat(10, 1) + 0.05 * torch.randn(10 * 16 * 20, 3, generator=torch.Generator().manual_seed(2))).to(d)
    ins = dict(x=c["x"].to(d), nodes=c["nodes"].to(d), ea=c["edge_attr"].to(d), v=c["v"].to(d), lm=c["loc_mean"].to(d))
    edges = [c["row"].to(d), c["col"].to(d)]
    t_out = c["t_out"].to(d)
    losses = {}
    for mode in ("eager", "graph"):
        m = make_egno(c, seed=4)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)

        def fn(x, nodes, ea, v, lm):
            xo, _, _ = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
            return ((xo - tgt) ** 2).mean()

        out = []
        if mode == "graph":
            step = nb.GraphedStep(fn, ins, opt, warmup=3)     # 3 eager steps (lazy optimizer state), then capture
            assert step.launches_per_replay > 10
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
    assert losses["graph"] == losses["eager"][3:], losses


def test_device_resident_rollouts_match_a_stepwise_loop_with_oracle_features_and_energies():
    """egno_rollout / segno_rollout (featurisation + energy kernels, no host synchronisation inside) against the
    reference's rollout structure written out with the oracle's featurisation and energy functions
    (main_simulation_simple_no.py:342-384, train_nbody.py:200-236, utils.py:126-144,175-195)."""
    d = dev()
    B, N, T, L = 6, 5, 4, 3
    # ---- EGNO, charged
    s = synth.sample_state("charged", B, N, seed=11)
    row, col = synth.canonical_edges(B, N)
    edges = [row.to(d), col.to(d)]
    torch.manual_seed(2)
    m = nb.EGNO(n_layers=2, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T, device=d)
    loc0, vel0, q = s["loc"].reshape(-1, 3).to(d), s["vel"].reshape(-1, 3).to(d), s["charges"].reshape(-1, 1).to(d)
    preds, e_last, e_all = nb.egno_rollout(m, loc0, vel0, q, edges, N, traj_len=L, dataset="charged")
    assert preds.shape == (L * T, B * N, 3) and e_last.shape == (L, B) and e_all.shape == (L * T, B)
    t_out = torch.arange(1, T + 1, device=d)[None].repeat(B, 1)
    loc, vel, ref_p, ref_e = loc0, vel0, [], []
    with torch.no_grad():
        for _ in range(L):
            x, nodes, ea, v, lm = synth.egno_features(loc.view(B, N, 3), vel.view(B, N, 3), q.view(B, N, 1), edges[0], edges[1])
            xo, vo, _ = m(x, nodes, edges, ea, v=v, loc_mean=lm, timesteps_out=t_out)
            xo, vo = xo.view(T, B * N, 3), vo.view(T, B * N, 3)
            ref_p.append(xo)
            for t in range(T):
                ref_e.append(O.energy_charged(xo[t].view(B, N, 3).cpu(), vo[t].view(B, N, 3).cpu(), q.view(B, N, 1).cpu()))
            loc, vel = xo[T - 1], vo[T - 1]
    assert rel_err(preds.cpu(), torch.cat(ref_p).cpu()) < 1e-5
    assert rel_err(e_all.cpu(), torch.stack(ref_e)) < 1e-4
    assert torch.equal(e_last, e_all.view(L, T, B)[:, T - 1])
    # ---- SEGNO, gravity
    s = synth.sample_state("gravity", B, N, seed=12)
    torch.manual_seed(3)
    sg = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True)
    loc0, vel0, mass = s["loc"].reshape(-1, 3).to(d), s["vel"].reshape(-1, 3).to(d), s["charges"].reshape(-1, 1).to(d)
    preds, en = nb.segno_rollout(sg, loc0, vel0, mass, edges, N, traj_len=L, num_steps=T, dataset="gravity")
    loc, vel, ref_p, ref_e = loc0, vel0, [], []
    with torch.no_grad():
        for _ in range(L):
            his, x, v, ea = synth.segno_features(loc.view(B, N, 3), vel.view(B, N, 3), mass.view(B, N, 1), edges[0], edges[1])
            xo, _, vo = sg(his, x, edges, v, ea, T=T)
            ref_p.append(xo)
            ref_e.append(O.energy_gravity(xo.view(B, N, 3).cpu(), vo.view(B, N, 3).cpu(), mass.view(B, N, 1).cpu()))
            loc, vel = xo, vo
    assert rel_err(preds.cpu(), torch.stack(ref_p).cpu()) < 1e-5
    assert rel_err(en.cpu(), torch.stack(ref_e)) < 1e-4


def test_flat_adam_matches_torch_adam_and_skips_inert_parameters():
    """FlatAdam (one fused launch over the flat parameter / gradient buffers) follows torch.optim.Adam step for step on
    EGNO; on SEGNO the never-used coord_mlp_vel tensors keep grad None (as in the reference) and are not updated."""
    d = dev()
    c = _egno_case(8, 5, 6, L=2, seed=21)
    tgt = torch.randn(6 * 8 * 5, 3, generator=torch.Generator().manual_seed(1)).to(d)
    finals = {}
    for kind in ("torch", "flat"):
        m = make_egno(c, seed=7)
        opt = (torch.optim.Adam if kind == "torch" else nb.FlatAdam)(m.parameters(), lr=2e-3, weight_decay=1e-4)
        for _ in range(4):
            opt.zero_grad(set_to_none=True)
            _, _, (xo, vo, ho) = run_egno(m, c, requires_grad=False)
            ((xo - tgt) ** 2).mean().backward()
            if kind == "flat":
                assert len(opt._runs(list(m.parameters()))) == 1   # parameters and gradients are each one flat buffer
            opt.step()
        finals[kind] = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).cpu()
    assert rel_err(finals["flat"], finals["torch"]) < 1e-5, rel_err(finals["flat"], finals["torch"])
    # SEGNO: inert tensors
    B, N = 4, 5
    s = synth.sample_state("gravity", B, N, seed=3)
    row, col = synth.canonical_edges(B, N)
    his, x, v, ea = synth.segno_features(s["loc"], s["vel"], s["charges"], row, col)
    sg = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True)
    before = {k: p.detach().clone() for k, p in sg.named_parameters()}
    opt = nb.FlatAdam(sg.parameters(), lr=1e-2, weight_decay=1e-2)
    xo, _, _ = sg(his.to(d), x.to(d), [row, col], v.to(d), ea.to(d), T=3)
    xo.square().mean().backward()
    opt.step()
    for k, p in sg.named_parameters():
        if "coord_mlp_vel" in k:
            assert p.grad is None and torch.equal(p.detach(), before[k]), k
        else:
            assert p.grad is not None and not torch.equal(p.detach(), before[k]), k


@pytest.mark.parametrize("name", SEGNO_MULTI_CASES)
def test_segno_multi_input_matches_reference_golden(name):
    """Several input frames (model.py:65-90): embedding of every observed frame, CUDA integration segments and the
    'sum' / attention merges between them (one autograd node, C calls only), against golden vectors of the reference."""
    dd, w, g = load_case(name)
    c = segno_multi_inputs_from_case(dd)
    d = dev()
    torch.manual_seed(1)
    m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True, multiple_agg=c["agg"])
    assert [k for k, _ in m.named_parameters()] == list(w.keys())
    m.load_state_dict(w)
    x = c["x"].to(d).requires_grad_(True)
    v = c["v"].to(d).requires_grad_(True)
    xo, ho, vo = m(c["his"].to(d), x, [c["row"], c["col"]], v, c["edge_attr"].to(d), T=c["T"], in_steps=c["in_steps"])
    assert rel_err(xo.cpu(), torch.tensor(dd["x_out"])) < TOL_OUT
    assert rel_err(vo.cpu(), torch.tensor(dd["v_out"])) < TOL_OUT
    assert rel_err(ho.cpu(), torch.tensor(dd["h_out"])) < TOL_OUT
    loss = (xo * torch.tensor(dd["Gx"], device=d)).sum() + (vo * torch.tensor(dd["Gv"], device=d)).sum() + \
        (ho * torch.tensor(dd["Gh"], device=d)).sum()
    loss.backward()
    assert rel_err(x.grad.cpu(), torch.tensor(dd["gx_in"])) < TOL_GRAD
    assert rel_err(v.grad.cpu(), torch.tensor(dd["gv_in"])) < TOL_GRAD
    for k, p in m.named_parameters():
        if k == "enc_attn_net.attn_mlp.2.bias":   # softmax is shift invariant: rounding noise in the reference too
            continue
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(g[k])
        assert rel_err(got, g[k]) < TOL_GRAD, k


@pytest.mark.parametrize("name", SEGNO_MULTI_CASES)
def test_segno_multi_input_launches_only_this_librarys_kernels(name):
    """VERDICT r01 item 10: the multi-input SEGNO forward + backward (embedding, segments, merges, gradient sums) must not
    run a single torch compute kernel — every kernel in the profiler's list is one of this library's (`k_*`)."""
    from torch.profiler import ProfilerActivity, profile
    dd, w, g = load_case(name)
    c = segno_multi_inputs_from_case(dd)
    d = dev()
    m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True, multiple_agg=c["agg"])
    m.load_state_dict(w)
    his, ea = c["his"].to(d), c["edge_attr"].to(d)
    G = [torch.tensor(dd[k], device=d) for k in ("Gx", "Gh", "Gv")]

    def run():
        x, v = c["x"].to(d).requires_grad_(True), c["v"].to(d).requires_grad_(True)
        torch.cuda.synchronize()
        return x, v

    x, v = run()
    out = m(his, x, [c["row"], c["col"]], v, ea, T=c["T"], in_steps=c["in_steps"])      # warm-up: flat views, edge check
    torch.autograd.backward(out, G)
    m.zero_grad(set_to_none=True)      # otherwise autograd would ADD the second gradient onto the first (a torch kernel)
    x, v = run()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        out = m(his, x, [c["row"], c["col"]], v, ea, T=c["T"], in_steps=c["in_steps"])
        torch.autograd.backward(out, G)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if getattr(e, "device_type", None) == torch.autograd.DeviceType.CUDA]
    kernels = [n for n in names if not n.lower().startswith(("memcpy", "memset"))]
    if not kernels:
        pytest.skip("the profiler recorded no device activity on this box")
    foreign = [n for n in kernels if not (n.startswith("k_") or n.startswith("void k_"))]
    assert not foreign, foreign
    assert any("k_segno_merge_fwd" in n for n in kernels) and any("k_segno_merge_bwd" in n for n in kernels)


@pytest.mark.parametrize("B,N,T,nin", [(4, 20, 10, 2), (2, 37, 6, 3)])
def test_egno_multi_input_vs_oracle_larger_graphs(B, N, T, nin):
    """Several input frames on the 20-body shape and on a graph that takes the blocked selector walk (N > 27), with
    per-trajectory output times; against the oracle restatement (pinned to the reference by the two golden cases)."""
    d = dev()
    g = torch.Generator().manual_seed(100 * N + nin)
    loc = torch.randn(nin, B, N, 3, generator=g) * 1.5
    vel = torch.randn(nin, B, N, 3, generator=g) * 0.3
    q = torch.randint(0, 2, (B, N, 1), generator=g).float() * 2 - 1
    row, col = O.canonical_edges(B, N)
    x, v, ea, nodes, lm = O.egno_features_multi(loc, vel, q, row, col)
    t_in = torch.arange(-nin + 1, 1)[None].repeat(B, 1)
    t_out = torch.stack([torch.sort(torch.randperm(2 * T, generator=g)[:T] + 1).values for _ in range(B)])
    torch.manual_seed(5)
    m = nb.EGNO(n_layers=2, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T,
                num_inputs=nin, device=d)
    w = {k: t.detach().cpu().clone() for k, t in m.state_dict().items()}
    xg = x.contiguous().to(d).requires_grad_(True)
    vg = v.contiguous().to(d).requires_grad_(True)
    xo, vo, ho = m(xg, nodes.contiguous().to(d), [row.to(d), col.to(d)], ea.contiguous().to(d), v=vg,
                   loc_mean=lm.contiguous().to(d), timesteps_in=t_in.to(d), timesteps_out=t_out.to(d))
    Gx, Gh = torch.randn(xo.shape, generator=g), torch.randn(ho.shape, generator=g) * 0.05
    ((xo * Gx.to(d)).sum() + (ho * Gh.to(d)).sum()).backward()
    p = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    xr, vr = x.clone().requires_grad_(True), v.clone().requires_grad_(True)
    xo_r, vo_r, ho_r = O.egno_forward_multi(p, xr, nodes, row, col, ea, vr, lm, t_in, t_out, n_layers=2, num_timesteps=T)
    ((xo_r * Gx).sum() + (ho_r * Gh).sum()).backward()
    assert rel_err(xo.cpu(), xo_r.detach()) < TOL_OUT
    assert rel_err(vo.cpu(), vo_r.detach()) < TOL_OUT
    assert rel_err(ho.cpu(), ho_r.detach()) < TOL_OUT
    assert rel_err(xg.grad.cpu(), xr.grad) < TOL_GRAD
    assert rel_err(vg.grad.cpu(), vr.grad) < TOL_GRAD
    # One-element parameters (the coordinate head's output bias) are sums of ~B*T*N*(N-1) signed per-edge terms; for
    # randn inputs layer 0's sum cancels to 0.34 against 10.7 in layer 1, and the fp32 SIMT variant (edge impl 0)
    # already sits 7e-4 from the fp32 oracle there.  Scale their tolerance by the largest same-named gradient across layers.
    def scale(k, ref):
        if ref.numel() > 1:
            return ref.abs().max()
        tail = k.split(".", 2)[-1]
        return max(float(p[j].grad.abs().max()) for j in p if j.endswith(tail) and p[j].grad is not None)
    param_grads_within_kink_budget(m, p, n_rows=T * B * N, tol=TOL_GRAD, scale=scale)


def test_blocked_selector_walk_is_deterministic_and_batch_independent():
    """N > 27 (blocked receiver x sender walk with shared-memory / TMEM accumulators): bitwise repeatable, and the
    result of a trajectory does not depend on what else is in the batch."""
    d = dev()
    c = _egno_case(3, 40, 4, L=1, seed=77)
    m = make_egno(c, seed=9)
    outs = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        x, v, (xo, vo, ho) = run_egno(m, c)
        (xo.square().sum() + ho.sum()).backward()
        outs.append([xo.detach().clone(), ho.detach().clone(), x.grad.clone()] + [p.grad.clone() for p in m.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*outs))
    # trajectory 0 alone: slice the batch of 3 (rows of graph 0 come first in every node / edge array)
    N, T = 40, 4
    row1, col1 = O.canonical_edges(1, N)
    c1 = dict(c, B=1, row=row1, col=col1, x=c["x"][:N], v=c["v"][:N], nodes=c["nodes"][:N], loc_mean=c["loc_mean"][:N],
              edge_attr=c["edge_attr"][:N * (N - 1)], t_out=c["t_out"][:1])
    with torch.no_grad():
        _, _, (xo1, vo1, ho1) = run_egno(m, c1, requires_grad=False)
    xo3 = outs[0][0].view(T, 3 * N, 3)[:, :N].reshape(-1, 3)
    ho3 = outs[0][1].view(T, 3 * N, -1)[:, :N].reshape(T * N, -1)
    assert rel_err(xo1.cpu(), xo3.cpu()) < 1e-6
    assert rel_err(ho1.cpu(), ho3.cpu()) < 1e-6


@pytest.mark.parametrize("only_first", [False, True])
def test_fused_trajectory_mse_matches_the_callers_loss(only_first):
    """nb.trajectory_mse (SURVEY 8f-4) on a model output at BASELINE sizes: loss, per-frame losses and the gradient that
    reaches the model against the oracle's restatement of main_simulation_simple_no.py:268-276 under autograd; both
    target layouts; bitwise reproducible."""
    dev = torch.device("cuda:0")
    T, B, N = 10, 256, 20
    g = torch.Generator().manual_seed(5)
    pred = torch.randn(T * B * N, 3, generator=g)
    tgt = torch.randn(B * N, T, 3, generator=g)
    pr = pred.clone().requires_grad_(True)
    loss_r, losses_r = O.trajectory_mse(pr, tgt, only_first)
    loss_r.backward()
    for target in (tgt.to(dev), tgt.reshape(B, N, T, 3).to(dev), tgt.transpose(0, 1).reshape(T * B * N, 3).contiguous().to(dev)):
        pd = pred.to(dev).requires_grad_(True)
        loss, losses = nb.trajectory_mse(pd, target, T, only_first)
        (3.0 * loss).backward()
        assert rel_err(losses.cpu(), losses_r.detach()) < 1e-5
        assert abs(loss.item() - loss_r.item()) < 1e-5 * abs(loss_r.item())
        assert rel_err(pd.grad.cpu(), 3.0 * pr.grad) < 1e-5
        loss2, _ = nb.trajectory_mse(pd.detach(), target, T, only_first)
        assert torch.equal(loss2, loss.detach())
    with pytest.raises(ValueError):
        nb.trajectory_mse(pred.to(dev), tgt.to(dev)[:, :5], T)


def test_segno_multi_input_under_data_parallel_matches_the_single_process_result():
    """enable_data_parallel() with several input frames (VERDICT r01 missing #7): the flat-bucket all-reduce of every
    integration segment plus dp_param for the torch-side parameters; with a world of one rank the result must be the
    single-process one bit for bit (the N > 1 arithmetic is covered on the CPU by tests/test_dp_gloo.py)."""
    import os
    import torch.distributed as dist

    dd, w, g = load_case("segno_n5_t6_in3_attn")
    c = segno_multi_inputs_from_case(dd)
    d = dev()
    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=d)
        created = True
    try:
        grads = {}
        for mode in ("single", "dp"):
            m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device=d, n_layers=8, recurrent=True, multiple_agg=c["agg"])
            m.load_state_dict(w)
            if mode == "dp":
                m.enable_data_parallel()
            xo, ho, vo = m(c["his"].to(d), c["x"].to(d), [c["row"], c["col"]], c["v"].to(d), c["edge_attr"].to(d), T=c["T"],
                           in_steps=c["in_steps"])
            (xo.square().sum() + ho.sum() + vo.square().sum()).backward()
            grads[mode] = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
        assert grads["single"].keys() == grads["dp"].keys() and len(grads["dp"]) >= 16
        for k in grads["single"]:
            assert torch.equal(grads["single"][k], grads["dp"][k]), k
    finally:
        if created:
            dist.destroy_process_group()


def test_peer_memory_data_parallel_matches_the_plain_optimizer_on_one_rank():
    """enable_data_parallel(peer_memory=True) + FlatAdam(peer_bucket=...): the gradient bucket lives in symmetric memory and
    the optimizer kernel sums the ranks' buckets itself (nb_adam_step_peers).  With a world of one rank the run must equal
    the plain FlatAdam run bit for bit, eagerly and under graph replay (2 / 8 ranks: tools/dp_check.py, bench.py)."""
    import os
    import torch.distributed as dist

    d = dev()
    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29534")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=d)
        created = True
    try:
        c = _egno_case(8, 5, 6, L=2, seed=21)
        tgt = torch.randn(6 * 8 * 5, 3, generator=torch.Generator().manual_seed(1)).to(d)
        finals = {}
        for kind in ("plain", "peer"):
            m = make_egno(c, seed=7)
            if kind == "peer":
                try:
                    m.enable_data_parallel(peer_memory=True)
                except Exception as e:      # symmetric memory unavailable on this box / build
                    pytest.skip(f"symmetric memory not available: {e}")
                assert m.peer_bucket is not None and m.peer_bucket.world == 1
            opt = nb.FlatAdam(m.parameters(), lr=2e-3, weight_decay=1e-4, peer_bucket=m.peer_bucket)
            for _ in range(3):
                opt.zero_grad(set_to_none=True)
                _, _, (xo, vo, ho) = run_egno(m, c, requires_grad=False)
                ((xo - tgt) ** 2).mean().backward()
                opt.step()
            finals[kind] = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).cpu()
        assert torch.equal(finals["plain"], finals["peer"])
    finally:
        if created:
            dist.destroy_process_group()
