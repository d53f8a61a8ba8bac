"""The configuration space the drop-in modules accept, held to the float64 oracle.

`EGNO(...)` / `SEGNO(...)` accept T <= 16, num_modes in [1, T/2+1], in_edge_nf 0..4, in_node_nf + time_emb_dim <= 128,
n_layers <= 32, SEGNO sub-step counts from 1 up and any recurrent / coords_weight; the kernels behind them specialise on
several of these (the T > 10 instantiation of the fused temporal convolution, the Nyquist / single-mode branches, the
selector edge kernels' graph packing, tail tiles and blocked walk, the per-layer offsets, the clamp masks).  One case
table drives two tiers:

  GPU tier  (pytest.mark.gpu): module -> C ABI -> sm_100a kernels.  Outputs within 1e-4 and input gradients within
            1e-3 of the float64 oracle (scale-relative); parameter gradients through
            helpers.param_grads_within_kink_budget (TimeConv's LeakyReLU kink, see test_gpu_parity.py).  SEGNO cases
            with N <= 27 run with the fused T-sub-step forward and with the stepwise kernels.
  CPU tier  the cases of at most ~200 nodes, through the host emulator build of the same sources (fp32 SIMT kernels,
            tests/emu_harness.py), at the emulator's 2e-5 bar against the same float64 oracle.

Every case checks that it reaches the path it is there for: the selector geometry (graph instances per unit, tail
tile rows, tail blocks, units per CTA) is recomputed here from sel_geom() in csrc/nbody_b200.cu, clamp cases measure
the saturated fraction in the oracle, and T > 10 cases check T.

Weights are the modules' own initial weights under torch.manual_seed, with TimeConv's spectral weights (1/64^2 scale at
init) multiplied by 20 so that the convolution of h moves the result, and the coordinate heads scaled up (SEGNO's last
layer has xavier gain 1e-3) so that the coordinate path is visible; clamp cases scale them further into saturation.
"""
from __future__ import annotations

import contextlib

import pytest
import torch

import no_node_comparison_b200 as nb
from no_node_comparison_b200 import synth
from oracle import nbody_oracle as O
from tests.helpers import param_grads_within_kink_budget, rel_err

TOL_OUT = 1e-4
TOL_GRAD = 1e-3
TOL_EMU = 2e-5            # fp32 SIMT kernels vs the float64 oracle (test_emu_kernels.py)
EMU_MAX_NODES = 200       # T*B*N of the cases the CPU tier runs (a few seconds each in the emulator) ...
EMU_MAX_LAYERS = 6        # ... and layers (about one second each, whatever the size)
TCONV_SCALE = 20.0
SAT_BAND = (0.05, 0.95)   # clamp cases: fraction of the clamped components that saturate
ENVELOPE = 30.0           # deep case: multiple of the fp32 oracle's own distance from float64

_EGNO = dict(model="egno", B=3, N=5, T=4, L=1, modes=2, in_node_nf=2, in_edge_nf=2, time_emb_dim=32, use_time_conv=True,
             num_inputs=1, coord_scale=1.0, vardt=False)
_SEGNO = dict(model="segno", B=4, N=5, T=4, in_node_nf=1, in_edge_nf=2, recurrent=True, coords_weight=1.0,
              coord_scale=200.0)


def _case(base, name, seed, **kw):
    c = dict(base, name=name, seed=seed, geom=None, clamp=False, long=False, envelope=False, emu=True)
    c.update(kw)
    return c


def egno(name, seed, **kw):
    return _case(_EGNO, name, seed, **kw)


def segno(name, seed, **kw):
    return _case(_SEGNO, name, seed, **kw)


CASES = [
    # --- EGNO temporal convolution: single mode, Nyquist at m = 1 (T = 2), the T > 10 instantiation, modes > 2
    egno("egno_T1_m1", 1, T=1, modes=1),
    egno("egno_T2_m2", 2, T=2, modes=2, L=2),
    egno("egno_T8_m1", 3, T=8, modes=1),
    egno("egno_T11_m2", 4, T=11, modes=2, B=2, long=True),
    egno("egno_T12_m1", 5, T=12, modes=1, B=2, long=True),
    egno("egno_T16_m2", 6, T=16, modes=2, B=2, long=True),
    egno("egno_T16_m9", 7, T=16, modes=9, B=2, long=True),
    egno("egno_T11_m6", 8, T=11, modes=6, B=2, long=True),
    egno("egno_T5_m5_clamped_to_3", 9, T=5, modes=5),
    egno("egno_no_time_conv", 10, use_time_conv=False, T=6, L=2),
    # --- EGNO features
    egno("egno_edge_nf0", 11, in_edge_nf=0),
    egno("egno_edge_nf1", 12, in_edge_nf=1),
    egno("egno_edge_nf3", 13, in_edge_nf=3),
    egno("egno_edge_nf4", 14, in_edge_nf=4),
    egno("egno_edge_nf3_blocked", 15, in_edge_nf=3, N=29, B=1, T=2, L=1, geom=dict(blk=1)),
    egno("egno_node1_temb16", 16, in_node_nf=1, time_emb_dim=16),
    egno("egno_node64_temb64", 17, in_node_nf=64, time_emb_dim=64),
    egno("egno_node3_temb64", 18, in_node_nf=3, time_emb_dim=64),
    # --- EGNO depth
    egno("egno_L6", 19, L=6, B=1, N=4, T=3),
    egno("egno_L32", 20, L=32, B=2, N=3, T=2, envelope=True),
    # --- EGNO several input frames: per-frame edge features of width 3, the T > 10 frame map, per-trajectory times
    egno("egno_in3_T12_ef3", 21, num_inputs=3, T=12, in_edge_nf=3, B=2, L=2, vardt=True, long=True),
    # --- selector geometry (one layer: the edge kernels are the subject)
    egno("egno_sel_N4_G6_partial", 22, N=4, B=13, T=1, L=1, geom=dict(blk=0, G=6, partial=True), emu=False),
    egno("egno_sel_N7_G3", 23, N=7, B=4, T=2, L=1, geom=dict(blk=0, G=3, partial=True), emu=False),
    egno("egno_sel_N8_G2", 24, N=8, B=3, T=3, L=1, geom=dict(blk=0, G=2, partial=True), emu=False),
    egno("egno_sel_N12_tail4", 25, N=12, B=2, T=2, L=1, geom=dict(blk=0, G=1, tail=4), emu=False),
    egno("egno_sel_N26_tail10", 26, N=26, B=1, T=2, L=1, geom=dict(blk=0, G=1, tail=10), emu=False),
    egno("egno_sel_N29_tail1", 27, N=29, B=2, T=2, L=1, geom=dict(blk=1, IB=4, tailI=1), emu=False),
    egno("egno_sel_N57_tails1_25", 28, N=57, B=1, T=2, L=1, geom=dict(blk=1, tailI=1, tailJ=25), emu=False),
    egno("egno_sel_N12_many_units", 29, N=12, B=300, T=2, L=1, geom=dict(blk=0, many_units=True), emu=False),
    egno("egno_sel_N29_many_units", 30, N=29, B=300, T=2, L=1, geom=dict(blk=1, many_units=True), emu=False),
    # --- EGNO clamp(+-100) of the per-node mean force, saturated
    egno("egno_clamp_N5", 31, N=5, B=4, T=3, L=1, coord_scale=4000.0, clamp=True, geom=dict(blk=0)),
    egno("egno_clamp_N29", 32, N=29, B=1, T=2, L=1, coord_scale=1600.0, clamp=True, geom=dict(blk=1)),
    # --- SEGNO
    segno("segno_nonrecurrent", 41, recurrent=False),
    segno("segno_cw0.5", 42, coords_weight=0.5),
    segno("segno_cw2", 43, coords_weight=2.0),
    segno("segno_node3", 44, in_node_nf=3),
    segno("segno_node64", 45, in_node_nf=64),
    segno("segno_edge_nf0", 46, in_edge_nf=0),
    segno("segno_edge_nf4", 47, in_edge_nf=4),
    segno("segno_edge_nf4_blocked", 48, in_edge_nf=4, N=29, B=1, T=3, geom=dict(blk=1)),
    segno("segno_T1", 49, T=1),
    segno("segno_T40", 50, T=40, B=2),
    segno("segno_sel_N4_G6_partial", 51, N=4, B=13, T=2, geom=dict(blk=0, G=6, partial=True), emu=False),
    segno("segno_sel_N7_G3", 52, N=7, B=4, T=2, geom=dict(blk=0, G=3, partial=True), emu=False),
    segno("segno_sel_N8_G2", 53, N=8, B=3, T=2, geom=dict(blk=0, G=2, partial=True), emu=False),
    segno("segno_sel_N12_tail4", 54, N=12, B=2, T=3, geom=dict(blk=0, G=1, tail=4), emu=False),
    segno("segno_sel_N26_tail10", 55, N=26, B=1, T=3, geom=dict(blk=0, G=1, tail=10), emu=False),
    segno("segno_sel_N29_tail1", 56, N=29, B=2, T=2, geom=dict(blk=1, IB=4, tailI=1), emu=False),
    segno("segno_sel_N57_tails1_25", 57, N=57, B=1, T=2, geom=dict(blk=1, tailI=1, tailJ=25), emu=False),
    segno("segno_sel_N12_many_units", 58, N=12, B=600, T=2, geom=dict(blk=0, many_units=True), emu=False),
    segno("segno_sel_N29_many_units", 59, N=29, B=300, T=2, geom=dict(blk=1, many_units=True), emu=False),
    # --- SEGNO clamp(+-100) of the per-edge rij * c, saturated
    segno("segno_clamp_N5", 61, N=5, B=4, T=3, coord_scale=1.5e5, clamp=True, geom=dict(blk=0)),
    segno("segno_clamp_N29", 62, N=29, B=1, T=2, coord_scale=2.0e6, clamp=True, geom=dict(blk=1)),
]


def _nodes(c):
    return (c["T"] if c["model"] == "egno" else 1) * c["B"] * c["N"]


def _emu_cases():
    """The emulator runs the SIMT edge tiles, not the selector kernels: the selector-geometry cases and the blocked walk
    (N > 27) are the GPU tier's alone."""
    return [c for c in CASES if c["emu"] and c["N"] <= 27 and _nodes(c) <= EMU_MAX_NODES and c.get("L", 1) <= EMU_MAX_LAYERS]


# ----------------------------------------------------------------------------------------------------- selector geometry
def sel_geom(N, n_gt):
    """sel_geom() of csrc/nbody_b200.cu: N <= 27 packs G graph instances (G*N <= 27 nodes, G*N(N-1) <= 128 rows for
    G > 1) into one unit of 128-row tiles; larger N walks IB receivers x JB senders blocks, one graph instance per unit."""
    if N > 27:
        best = None
        for ib in range(1, 33):
            jb = min(128 // ib, 32, N)
            if ib + jb > 54 or jb < 1:
                continue
            tiles = -(-N // ib) * -(-N // jb)
            if best is None or tiles < best[0]:
                best = (tiles, ib, jb)
        _, ib, jb = best
        return dict(blk=1, G=1, units=n_gt, IB=ib, JB=jb, tailI=N - (-(-N // ib) - 1) * ib,
                    tailJ=N - (-(-N // jb) - 1) * jb)
    G = max(1, min(128 // (N * (N - 1)), 27 // N))
    return dict(blk=0, G=G, units=-(-n_gt // G), tail=G * N * (N - 1) % 128, partial=n_gt % G != 0)


def check_geometry(c, sms=None):
    if c["geom"] is None:
        return
    g = sel_geom(c["N"], (c["T"] if c["model"] == "egno" else 1) * c["B"])
    for k, want in c["geom"].items():
        if k == "many_units":
            # the backward and the fused SEGNO forward run min(units, SMs) persistent CTAs, the edge forward
            # min(units, 2 x SMs): past 2 x SMs units every backward CTA walks at least two graph instances, so the
            # per-unit accumulators must be reset between them
            if sms is not None:
                assert g["units"] > 2 * sms, (g, sms)
        else:
            assert g[k] == want, (c["name"], k, g)


# ----------------------------------------------------------------------------------------------------- inputs and weights
def _widen(t, n, gen):
    """The physical feature columns, then seeded uniform columns up to width n (or the first n columns)."""
    w = t.shape[-1]
    if n <= w:
        return t[..., :n].contiguous()
    return torch.cat([t, torch.rand(t.shape[:-1] + (n - w,), generator=gen)], dim=-1).contiguous()


def make_inputs(c):
    B, N, T = c["B"], c["N"], c["T"]
    gen = torch.Generator().manual_seed(1000 + c["seed"])
    row, col = synth.canonical_edges(B, N)
    d = dict(row=row, col=col)
    if c["model"] == "segno":
        s = synth.sample_state("gravity", B, N, c["seed"])
        his, x, v, ea = synth.segno_features(s["loc"], s["vel"], s["charges"], row, col)
        d.update(his=_widen(his, c["in_node_nf"], gen), x=x, v=v, ea=_widen(ea, c["in_edge_nf"], gen))
        return d
    nin = c["num_inputs"]
    if nin == 1:
        s = synth.sample_state("charged", B, N, c["seed"])
        x, nodes, ea, v, lm = synth.egno_features(s["loc"], s["vel"], s["charges"], row, col)
        d.update(t_in=None)
    else:
        frames = [synth.sample_state("charged", B, N, c["seed"] + 97 * i) for i in range(nin)]
        loc = torch.stack([f["loc"] for f in frames])
        vel = torch.stack([f["vel"] for f in frames])
        x, v, ea, nodes, lm = O.egno_features_multi(loc, vel, frames[0]["charges"], row, col)
        x, v, lm = x.contiguous(), v.contiguous(), lm.contiguous()
        d.update(t_in=torch.arange(-nin + 1, 1)[None].repeat(B, 1))
    if c["vardt"]:
        t_out = torch.stack([torch.sort(torch.randperm(2 * T, generator=gen)[:T] + 1).values for _ in range(B)])
    else:
        t_out = torch.arange(1, T + 1)[None].repeat(B, 1)
    d.update(x=x, v=v, lm=lm, nodes=_widen(nodes, c["in_node_nf"], gen), ea=_widen(ea, c["in_edge_nf"], gen), t_out=t_out)
    return d


def make_model(c, device):
    torch.manual_seed(c["seed"])
    if c["model"] == "egno":
        m = nb.EGNO(n_layers=c["L"], in_node_nf=c["in_node_nf"], in_edge_nf=c["in_edge_nf"], hidden_nf=64, with_v=True,
                    use_time_conv=c["use_time_conv"], num_modes=c["modes"], num_timesteps=c["T"],
                    time_emb_dim=c["time_emb_dim"], num_inputs=c["num_inputs"], varDT=c["vardt"], device=device)
        with torch.no_grad():
            for tc in (m.time_conv_modules if c["use_time_conv"] else []):
                tc.t_conv.weights1.mul_(TCONV_SCALE)
            for layer in m.layers:
                layer.coord_net.mlp[2].weight.mul_(c["coord_scale"])
    else:
        m = nb.SEGNO(in_node_nf=c["in_node_nf"], in_edge_nf=c["in_edge_nf"], hidden_nf=64, device=device, n_layers=8,
                     recurrent=c["recurrent"], coords_weight=c["coords_weight"])
        with torch.no_grad():
            m.module.coord_mlp[2].weight.mul_(c["coord_scale"])
    return m


def cotangents(c):
    gen = torch.Generator().manual_seed(7 + c["seed"])
    n = _nodes(c)
    return dict(x=torch.randn(n, 3, generator=gen), v=torch.randn(n, 3, generator=gen),
                h=0.05 * torch.randn(n, 64, generator=gen))


# ----------------------------------------------------------------------------------------------------- the oracle
@contextlib.contextmanager
def _recording_segment_means(rec):
    """The oracle's clamp sits on the per-node mean force (EGNO: clamp of the mean) or on the per-edge terms that enter
    the mean (SEGNO: mean of the clamped rij * c); both pass through O.segment_mean, which this records."""
    orig = O.segment_mean

    def seg_mean(data, idx, n):
        out = orig(data, idx, n)
        rec.append((data.detach(), out.detach()))
        return out

    O.segment_mean = seg_mean
    try:
        yield
    finally:
        O.segment_mean = orig


def oracle(c, w, inp, G, dtype=torch.float64):
    """Outputs, input gradients and parameter leaves (with .grad) of the oracle in `dtype`, and the fraction of the
    clamped components that saturate."""
    cast = lambda t: None if t is None else t.to(dtype)
    p = {k: t.detach().to(dtype).requires_grad_(True) for k, t in w.items()}
    x = inp["x"].to(dtype).requires_grad_(True)
    v = inp["v"].to(dtype).requires_grad_(True)
    rec = []
    with _recording_segment_means(rec):
        if c["model"] == "egno":
            kw = dict(n_layers=c["L"], num_timesteps=c["T"], time_emb_dim=c["time_emb_dim"])
            if c["num_inputs"] == 1:
                xo, vo, ho = O.egno_forward(p, x, cast(inp["nodes"]), inp["row"], inp["col"], cast(inp["ea"]), v,
                                            cast(inp["lm"]), inp["t_out"], use_time_conv=c["use_time_conv"], **kw)
            else:
                xo, vo, ho = O.egno_forward_multi(p, x, cast(inp["nodes"]), inp["row"], inp["col"], cast(inp["ea"]), v,
                                                  cast(inp["lm"]), inp["t_in"], inp["t_out"], **kw)
        else:
            xo, ho, vo = O.segno_forward(p, cast(inp["his"]), x, inp["row"], inp["col"], v, cast(inp["ea"]), c["T"],
                                         recurrent=c["recurrent"], coords_weight=c["coords_weight"])
    ((xo * G["x"].to(dtype)).sum() + (vo * G["v"].to(dtype)).sum() + (ho * G["h"].to(dtype)).sum()).backward()
    if c["model"] == "egno":   # clamp(mean): components of the per-node mean force beyond +-100
        sat = torch.cat([o.reshape(-1) for _, o in rec]).abs().gt(100.0).double().mean().item()
    else:                      # mean(clamp): per-edge rij * c at +-100 (clamped already)
        sat = torch.cat([d.reshape(-1) for d, _ in rec]).abs().ge(100.0).double().mean().item()
    out = dict(x=xo.detach(), v=vo.detach(), h=ho.detach(), gx=x.grad, gv=v.grad)
    return out, p, sat


def weights_of(m):
    return {k: t.detach().cpu().clone() for k, t in m.named_parameters()}


# ----------------------------------------------------------------------------------------------------- comparison
def _grad_scale(p):
    """Scale of a parameter gradient: its largest entry.  A one-element tensor (the coordinate head's output bias) is a
    sum of signed per-edge terms that can cancel far below their size; it takes the scale of the same Linear's weight
    gradient, which sums the same per-edge terms times O(1) activations."""
    def scale(k, ref):
        s = float(ref.abs().max())
        if ref.numel() == 1 and k.endswith(".bias"):
            sib = p.get(k[:-len("bias")] + "weight")
            if sib is not None and sib.grad is not None:
                s = max(s, float(sib.grad.abs().max()))
        return max(s, 1e-30)
    return scale


def check_case(c, got, m, ref, p, tol_out, tol_grad, w, inp, G, label):
    """got / ref: outputs and input gradients; m: the module whose .grad fields hold the parameter gradients under
    test; p: the oracle's parameter leaves."""
    if c["envelope"]:
        # deep stacks are conditioned worse than one layer: hold the result to a multiple of the fp32 oracle's own
        # distance from float64 (test_gpu_curves.py, test_egno_100_body_config5_against_the_oracle)
        r32, p32, _ = oracle(c, w, inp, G, dtype=torch.float32)
        noise_out = max(rel_err(r32[k], ref[k]) for k in ("x", "v", "h"))
        noise_grad = max([rel_err(r32[k], ref[k]) for k in ("gx", "gv")] +
                         [rel_err(p32[k].grad, p[k].grad) for k in p if p[k].grad is not None])
        print(f"  fp32 oracle vs float64: outputs {noise_out:.1e}, gradients {noise_grad:.1e}")
        tol_out, tol_grad = max(tol_out, ENVELOPE * noise_out), max(tol_grad, ENVELOPE * noise_grad)
    errs = {k: rel_err(got[k], ref[k]) for k in ("x", "v", "h", "gx", "gv")}
    scale = _grad_scale(p)
    errs["params"] = 0.0
    for k, q in m.named_parameters():
        r = p[k].grad if p[k].grad is not None else torch.zeros(q.shape, dtype=torch.float64)
        g = q.grad.cpu() if q.grad is not None else torch.zeros(q.shape)
        errs["params"] = max(errs["params"], float((g.double() - r).abs().max() / scale(k, r)))
    print(f"{label} {c['name']}: worst rel err " + " ".join(f"{k}={e:.1e}" for k, e in errs.items()) +
          f" (bars {tol_out:.0e} / {tol_grad:.0e})")
    for k in ("x", "v", "h"):
        assert errs[k] < tol_out, (c["name"], k, errs)
    for k in ("gx", "gv"):
        assert errs[k] < tol_grad, (c["name"], k, errs)
    param_grads_within_kink_budget(m, p, n_rows=_nodes(c), tol=tol_grad, scale=scale)


def check_paths(c, m, sat, sms=None):
    check_geometry(c, sms)
    if c["clamp"]:
        print(f"  saturated fraction of the clamped components: {sat:.3f}")
        assert SAT_BAND[0] <= sat <= SAT_BAND[1], (c["name"], sat)
    if c["long"]:
        assert c["T"] > 10 and m.num_timesteps > 10
    if c["model"] == "egno" and c["T"] == 5:
        assert m.num_modes == 3 and c["modes"] > 3          # the constructor clamp at T = 5 (egno.py:26)


# ----------------------------------------------------------------------------------------------------- CPU tier
def _emu_run(c, m, inp, G):
    from tests import emu_harness as E

    params = E.flat_params({k: t.detach().numpy() for k, t in m.named_parameters()}, [k for k, _ in m.named_parameters()])
    n = lambda t: None if t is None else t.numpy()
    if c["model"] == "egno":
        cfg = dict(B=c["B"], N=c["N"], T=c["T"], n_layers=c["L"], num_modes=m.num_modes if c["use_time_conv"] else 1,
                   in_node_nf=c["in_node_nf"], in_edge_nf=c["in_edge_nf"], time_emb_dim=c["time_emb_dim"],
                   use_time_conv=int(c["use_time_conv"]), num_inputs=c["num_inputs"])
        r = E.egno_run(cfg, params, n(inp["x"]), n(inp["nodes"]), n(inp["ea"]), n(inp["v"]), n(inp["lm"]), n(inp["t_out"]),
                       n(G["x"]), n(G["v"]), n(G["h"]), t_in=n(inp["t_in"]))
    else:
        cfg = dict(B=c["B"], N=c["N"], T=c["T"], in_node_nf=c["in_node_nf"], in_edge_nf=c["in_edge_nf"],
                   recurrent=int(c["recurrent"]), coords_weight=c["coords_weight"])
        r = E.segno_run(cfg, params, n(inp["his"]), n(inp["x"]), n(inp["v"]), n(inp["ea"]), n(G["x"]), n(G["h"]), n(G["v"]))
    off = 0
    for _, q in m.named_parameters():
        q.grad = torch.tensor(r["grad_params"][off:off + q.numel()]).view_as(q)
        off += q.numel()
    assert off == r["grad_params"].size
    return dict(x=torch.tensor(r["x_out"]), v=torch.tensor(r["v_out"]), h=torch.tensor(r["h_out"]),
                gx=torch.tensor(r["gx_in"]).view(inp["x"].shape), gv=torch.tensor(r["gv_in"]).view(inp["v"].shape))


@pytest.mark.parametrize("c", _emu_cases(), ids=lambda c: c["name"])
def test_config_space_emulated_kernels_vs_float64_oracle(c):
    """The host-side layout (parameter offsets, saved-state strides, frame maps) and the fp32 SIMT kernels for every
    axis of the table, at the shapes the emulator runs in seconds."""
    m = make_model(c, "cpu")
    w = weights_of(m)
    inp = make_inputs(c)
    G = cotangents(c)
    ref, p, sat = oracle(c, w, inp, G)
    check_paths(c, m, sat)
    got = _emu_run(c, m, inp, G)
    check_case(c, got, m, ref, p, TOL_EMU, TOL_EMU, w, inp, G, "emulator")


def test_emulator_tier_covers_every_axis():
    """The CPU tier is a restriction by size only: every axis of the table keeps at least one case there."""
    names = {c["name"] for c in _emu_cases()}
    for need in ("egno_T1_m1", "egno_T2_m2", "egno_T16_m9", "egno_T11_m6", "egno_no_time_conv", "egno_edge_nf0",
                 "egno_edge_nf4", "egno_node64_temb64", "egno_L6", "egno_in3_T12_ef3", "egno_clamp_N5",
                 "segno_nonrecurrent", "segno_cw2", "segno_node64", "segno_edge_nf0", "segno_T40", "segno_clamp_N5"):
        assert need in names, need


# ----------------------------------------------------------------------------------------------------- GPU tier
def _cuda_run(c, m, inp, G):
    d = torch.device("cuda:0")
    x = inp["x"].to(d).requires_grad_(True)
    v = inp["v"].to(d).requires_grad_(True)
    edges = [inp["row"].to(d), inp["col"].to(d)]
    if c["model"] == "egno":
        t_in = None if inp["t_in"] is None else inp["t_in"].to(d)
        xo, vo, ho = m(x, inp["nodes"].to(d), edges, inp["ea"].to(d), v=v, loc_mean=inp["lm"].to(d),
                       timesteps_in=t_in, timesteps_out=inp["t_out"].to(d))
    else:
        xo, ho, vo = m(inp["his"].to(d), x, edges, v, inp["ea"].to(d), T=c["T"])
    ((xo * G["x"].to(d)).sum() + (vo * G["v"].to(d)).sum() + (ho * G["h"].to(d)).sum()).backward()
    return dict(x=xo.detach().cpu(), v=vo.detach().cpu(), h=ho.detach().cpu(), gx=x.grad.cpu(), gv=v.grad.cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=lambda c: c["name"])
def test_config_space_cuda_vs_float64_oracle(c):
    """Module -> C ABI -> sm_100a kernels (tcgen05 selector edge kernels, fused node kernels, tensor-core GEMMs, fused
    temporal convolution, fused SEGNO forward) for every case of the table."""
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    d = torch.device("cuda:0")
    inp = make_inputs(c)
    G = cotangents(c)
    m = make_model(c, d)
    w = weights_of(m)
    ref, p, sat = oracle(c, w, inp, G)
    check_paths(c, m, sat, sms=torch.cuda.get_device_properties(0).multi_processor_count)
    if c["model"] == "egno" or c["N"] > 27:
        got = _cuda_run(c, m, inp, G)
        check_case(c, got, m, ref, p, TOL_OUT, TOL_GRAD, w, inp, G, "cuda")
        return
    lib = nb.load_library()
    for fused in (1, 0):       # the fused T-sub-step forward and the stepwise kernels, each against the oracle
        assert lib.nb_set_segno_fused(fused) == 0
        try:
            m.zero_grad(set_to_none=True)
            got = _cuda_run(c, m, inp, G)
            check_case(c, got, m, ref, p, TOL_OUT, TOL_GRAD, w, inp, G, f"cuda fused={fused}")
        finally:
            lib.nb_set_segno_fused(1)
    assert lib.nb_get_segno_fused() == 1
