import sys, torch
sys.path.insert(0, '.')
import no_node_comparison_b200 as nb
from no_node_comparison_b200 import synth
from oracle import nbody_oracle as O
from tests.helpers import rel_err
DEV = torch.device('cuda:0')
lib = nb.load_library()
def run(B, N, T, L, seed, kind='charged'):
    s = synth.sample_state(kind, B, N, seed)
    row, col = synth.canonical_edges(B, N)
    x, nodes, ea, v, lm = synth.egno_features(s["loc"], s["vel"], s["charges"], row, col)
    t_out = torch.arange(1, T + 1)[None].repeat(B, 1)
    torch.manual_seed(1)
    m = nb.EGNO(n_layers=L, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, num_timesteps=T, device=DEV)
    p = {k: t.detach().cpu().clone() for k, t in m.named_parameters()}
    with torch.no_grad():
        xo_r, vo_r, ho_r = O.egno_forward(p, x, nodes, row, col, ea, v, lm, t_out, n_layers=L, num_timesteps=T)
        pd = {k: t.double() for k, t in p.items()}
        xo_d, vo_d, ho_d = O.egno_forward(pd, x.double(), nodes.double(), row, col, ea.double(), v.double(), lm.double(), t_out, n_layers=L, num_timesteps=T)
    print(f"B={B} N={N} T={T} L={L}: oracle fp32 vs fp64: x {rel_err(xo_r, xo_d):.1e} h {rel_err(ho_r, ho_d):.1e}; |x|max {xo_d.abs().max():.2f} |x-x0|max {(xo_d - x.double().repeat(T,1)).abs().max():.2f}")
    for ei, ni in ((2, 1), (0, 0), (2, 0), (0, 1)):
        lib.nb_set_edge_impl(ei); lib.nb_set_node_impl(ni)
        with torch.no_grad():
            xo, vo, ho = m(x.to(DEV), nodes.to(DEV), [row.to(DEV), col.to(DEV)], ea.to(DEV), v=v.to(DEV), loc_mean=lm.to(DEV), timesteps_out=t_out.to(DEV))
        print(f"   edge_impl {ei} node_impl {ni}: vs fp32 oracle x {rel_err(xo.cpu(), xo_r):.1e} h {rel_err(ho.cpu(), ho_r):.1e} | vs fp64 x {rel_err(xo.cpu(), xo_d):.1e} h {rel_err(ho.cpu(), ho_d):.1e}")
    lib.nb_set_edge_impl(2); lib.nb_set_node_impl(1)
run(4, 100, 10, 4, 6)
run(4, 100, 10, 1, 6)
run(8, 20, 10, 4, 6)
run(4, 50, 10, 4, 6)
