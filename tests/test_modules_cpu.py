"""Host-side behaviour of the drop-in modules (no GPU): constructor / state_dict compatibility with the
reference's checkpoints, error behaviour, and the flat parameter packing."""
import pytest
import torch

import no_node_comparison_b200 as nb
from no_node_comparison_b200.functional import _EdgeCache, _ParamPack
from oracle import nbody_oracle as O
from tests.helpers import EGNO_CASES, EGNO_MULTI_CASES, SEGNO_CASES, SEGNO_MULTI_CASES, load_case


def _egno(**kw):
    args = dict(n_layers=4, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, flat=False, norm=False,
                num_modes=2, num_timesteps=8, time_emb_dim=32, num_inputs=1, device="cpu")
    args.update(kw)
    return nb.EGNO(**args)


def test_egno_loads_reference_checkpoint_names_and_shapes():
    _, w, _ = load_case("egno_n5_t8")
    m = _egno()
    assert [k for k, _ in m.named_parameters()] == list(w.keys())        # also the C-ABI flat layout order
    m.load_state_dict(w, strict=True)
    for k, p in m.state_dict().items():
        assert torch.equal(p, w[k])
    assert sum(p.numel() for p in m.parameters()) == 201736               # SURVEY.md §8a1
    assert m.num_timesteps == 8


def test_segno_loads_reference_checkpoint_names_and_shapes():
    _, w, _ = load_case("segno_n5_t10")
    m = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", n_layers=8, recurrent=True,
                 norm_diff=False, tanh=False)
    assert [k for k, _ in m.named_parameters()] == list(w.keys())
    m.load_state_dict(w, strict=True)
    assert sum(p.numel() for p in m.parameters()) == 33602                # SURVEY.md §8a9


def test_same_seed_gives_reference_initial_weights():
    """The weights of every golden case are the reference modules' initial weights under torch.manual_seed(1)
    (tests/golden/make_golden.py); the drop-in modules must draw the same values in the same order."""
    for name in EGNO_CASES + EGNO_MULTI_CASES:
        d, w, _ = load_case(name)
        T, n_layers, num_modes = (int(v) for v in d["meta"][2:5])
        num_inputs = int(d["meta"][5]) if len(d["meta"]) > 5 else 1
        torch.manual_seed(1)
        m = _egno(n_layers=n_layers, num_modes=num_modes, num_timesteps=T, num_inputs=num_inputs, varDT="vardt" in name)
        sd = m.state_dict()
        assert list(sd) == list(w) and all(torch.equal(sd[k], w[k]) for k in w), name
    for name in SEGNO_CASES + SEGNO_MULTI_CASES:
        d, w, _ = load_case(name)
        agg = None if "agg" not in d else ("sum" if int(d["agg"][0]) == 0 else "attn")
        torch.manual_seed(1)
        # constructor defaults for norm_diff / tanh: the golden modules were built with both False
        s = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", n_layers=8, recurrent=True, multiple_agg=agg)
        sd = s.state_dict()
        assert list(sd) == list(w) and all(torch.equal(sd[k], w[k]) for k in w), name


def test_num_modes_clamp_matches_reference_ctor():
    assert _egno(num_timesteps=5, num_modes=5).num_modes == 3       # egno.py:26
    assert _egno(num_timesteps=2, num_modes=4).num_modes == 2
    assert _egno(num_timesteps=10, num_modes=2, fix_out_size=True).num_timesteps == 10


def test_unsupported_configurations_raise():
    with pytest.raises(ValueError):
        _egno(hidden_nf=32)
    with pytest.raises(ValueError):
        _egno(with_v=False)
    with pytest.raises(ValueError):
        _egno(num_inputs=0)
    # several input frames: two time embeddings feed the embedding Linear (egno.py:13-16)
    assert _egno(num_inputs=2).embedding.weight.shape == (64, 2 + 2 * 32)
    with pytest.raises(ValueError):
        nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, tanh=True)
    # norm_diff=True would divide coord_diff by sqrt(radial) + 1 (EGNN's coord2radial): refused, not silently ignored
    with pytest.raises(ValueError, match="norm_diff"):
        nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, norm_diff=True)


def test_cpu_tensors_are_rejected_no_fallback():
    """The product path has no CPU fallback: host tensors raise instead of silently computing elsewhere."""
    m = _egno()
    B, N, T = 2, 5, 8
    row, col = O.canonical_edges(B, N)
    x = torch.randn(B * N, 3)
    with pytest.raises(ValueError, match="CUDA"):
        m(x, torch.randn(B * N, 2), [row, col], torch.randn(B * N * (N - 1), 2), v=torch.randn(B * N, 3),
          loc_mean=torch.zeros(B * N, 3), timesteps_out=torch.arange(1, T + 1)[None].repeat(B, 1))
    s = nb.SEGNO(in_node_nf=1, in_edge_nf=2, hidden_nf=64, device="cpu", recurrent=True)
    with pytest.raises(ValueError, match="CUDA"):
        s(torch.randn(B * N, 1), x, [row, col], torch.randn(B * N, 3), torch.randn(B * N * (N - 1), 2), T=3)


def test_edge_validation_on_host_lists():
    c = _EdgeCache()
    row, col = O.canonical_edges(3, 5)
    c.validate([row, col], 3, 5, torch.device("cpu"))
    c.validate(torch.stack([row, col]), 3, 5, torch.device("cpu"))           # [2,E] tensor form (train_nbody.py:79)
    bad = col.clone()
    bad[3], bad[4] = col[4], col[3]
    with pytest.raises(ValueError, match="canonical"):
        c.validate([row, bad], 3, 5, torch.device("cpu"))
    with pytest.raises(ValueError):
        c.validate([row[:-1], col[:-1]], 3, 5, torch.device("cpu"))


def test_param_pack_keeps_views_through_optimizer_and_load():
    m = _egno(n_layers=1)
    pack = _ParamPack(m)
    n = sum(p.numel() for p in m.parameters())
    flat, ps = pack.flat_params(n, torch.device("cpu"))
    assert flat.numel() == n and all(p.data_ptr() >= flat.data_ptr() for p in ps)
    # order == named_parameters == C layout
    o = 0
    for p in ps:
        assert torch.equal(flat[o:o + p.numel()].view(p.shape), p.detach())
        o += p.numel()
    opt = torch.optim.Adam(m.parameters(), lr=1e-2)
    for p in m.parameters():
        p.grad = torch.ones_like(p)
    opt.step()
    flat2, _ = pack.flat_params(n, torch.device("cpu"))
    assert flat2.data_ptr() == flat.data_ptr()                               # still the same storage
    assert torch.equal(flat2[:8], ps[0].detach().reshape(-1)[:8])
    sd = {k: torch.zeros_like(v) for k, v in m.state_dict().items()}
    m.load_state_dict(sd)
    assert float(pack.flat_params(n, torch.device("cpu"))[0].abs().sum()) == 0.0
    m.double().float()                                                        # storage replaced -> repacked
    flat3, _ = pack.flat_params(n, torch.device("cpu"))
    assert flat3.data_ptr() != flat.data_ptr()


def test_helper_apis_refuse_cpu_tensors_and_bad_shapes():
    """trajectory_mse / simulate_* have no CPU path: host tensors and malformed arguments raise before any launch."""
    import no_node_comparison_b200 as nb
    T, R = 4, 10
    pred, tgt = torch.randn(T * R, 3), torch.randn(R, T, 3)
    with pytest.raises(ValueError, match="CUDA"):
        nb.trajectory_mse(pred, tgt, T)
    with pytest.raises(ValueError):
        nb.trajectory_mse(torch.randn(T * R + 1, 3), tgt, T)          # rows not a multiple of T
    with pytest.raises(ValueError):
        nb.trajectory_mse(pred, torch.randn(R, T + 1, 3), T)          # target frame count
    with pytest.raises(ValueError):
        nb.trajectory_mse(pred, tgt.requires_grad_(True), T)          # no gradient w.r.t. the target
    loc0 = torch.randn(2, 3, 5, dtype=torch.float64)
    with pytest.raises(ValueError, match="CUDA"):
        nb.simulate_charged(loc0, loc0.clone(), torch.ones(2, 5, dtype=torch.float64), 200, 100)
    with pytest.raises(ValueError):
        nb.simulate_charged(loc0, loc0.clone(), torch.ones(2, 5, dtype=torch.float64), 250, 100)   # T % sample_freq
    with pytest.raises(ValueError, match="CUDA"):
        nb.simulate_gravity(torch.randn(2, 5, 3, dtype=torch.float64), torch.randn(2, 5, 3, dtype=torch.float64),
                            torch.ones(2, 5, dtype=torch.float64), 100, 100)
