import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import no_node_comparison_b200 as nb
import tests.test_gpu_parity as T
lib = nb.load_library()
c = T._egno_case(8, 20, 10, L=4, seed=28)
res = {}
for ni in (0, 1):
    lib.nb_set_node_impl(ni)
    m = T.make_egno(c)
    x, v, (xo, vo, ho) = T.run_egno(m, c)
    gen = torch.Generator().manual_seed(3)
    Gx, Gh = torch.randn(xo.shape, generator=gen), torch.randn(ho.shape, generator=gen) * 0.05
    ((xo * Gx.cuda()).sum() + (ho * Gh.cuda()).sum()).backward()
    res[ni] = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters() if p.grad is not None}
    res[ni]['xo'] = xo.detach().cpu(); res[ni]['ho'] = ho.detach().cpu(); res[ni]['gx'] = x.grad.cpu()
for k in res[0]:
    a, b = res[0][k], res[1][k]
    e = (a - b).abs().max().item() / (a.abs().max().item() + 1e-30)
    if e > 2e-4:
        d = (a - b).abs()
        idx = torch.nonzero(d > 0.3 * d.max())
        print(k, 'rel', e, 'max', a.abs().max().item(), 'n_big', len(idx), idx[:12].tolist())
print('done')
