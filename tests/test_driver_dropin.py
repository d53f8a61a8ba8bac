"""Driver-level drop-in proof (SURVEY.md §8c "driver-level oracle"; VERDICT r01 missing #3).

The reference's unmodified `run_epoch` / `rollout_fn` (EGNO/main_simulation_simple_no.py:190-384,
SEGNO/train_nbody.py:57-236) with the reference's own dataset classes, loss, Adam and numpy energies drive

  * the reference's modules on the CPU  and  * `no_node_comparison_b200.EGNO / SEGNO` on the GPU     (-m gpu)
  * the reference's modules  and  * the oracle restatement wrapped as a module                        (not gpu)

on the same simulated data set and the same initial weights; training losses, validation loss, rollout predictions,
per-frame test MSE and energy curves must agree.  The reference is imported through oracle/ref_loader.py (the
original checkout, or the unmodified copy oracle/make_ref.py installs into oracle/_ref); the tests skip without it.

Tolerances (fp32): a 1e-5 relative perturbation of the weights moves these quantities by 1e-5 .. 6e-5 (measured with
the reference on the CPU), the CUDA path's own forward error is <= 2e-5; the bounds below leave a 20-50x margin.
"""
from __future__ import annotations

import pytest
import torch

from oracle import nbody_oracle as O
from oracle import ref_loader as RL
from tests import dataset_factory as DF
from tests import driver_harness as H

needs_ref = pytest.mark.skipif(not RL.reference_available(), reason="reference not installed (run oracle/make_ref.py)")

EGNO_KW = dict(n_layers=4, in_node_nf=2, in_edge_nf=2, hidden_nf=64, with_v=True, num_modes=2, time_emb_dim=32)
SEGNO_KW = dict(in_node_nf=1, in_edge_nf=2, hidden_nf=64, n_layers=8, recurrent=True, norm_diff=False, tanh=False)


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-12)


def _compare(ours, ref, what, per_call=1):
    for i, (a, b) in enumerate(zip(ours["train"], ref["train"])):
        assert _rel(a, b) < 2e-3, f"{what}: train loss of epoch {i}: {a} vs {b}"
    assert _rel(ours["valid"], ref["valid"]) < 2e-3, f"{what}: validation loss {ours['valid']} vs {ref['valid']}"
    assert ours["preds"].shape == ref["preds"].shape
    # The rollout is an iterated map of a model that has seen two epochs: the difference of the first call (the 1e-5 of
    # a forward pass plus the slightly different trained weights) grows 4-5x per call on every path (measured: 1.6e-5,
    # 2.2e-4, 1.2e-3, 3.9e-3, 9.2e-3 for SEGNO, gravity, N=5; see tests/test_gpu_curves.py for the measured envelope).
    # The first call already carries the weight difference of two epochs of training (1.3e-4 .. 2.3e-4 observed; the
    # multi-threaded CPU reference is itself not bitwise repeatable).  Bounds per call k: 5e-4 * 6^k, capped at 0.25.
    F = ours["preds"].shape[1]          # emitted frames; `per_call` of them per model call
    tol = lambda k: min(5e-4 * 6.0 ** (k // per_call), 0.25)
    scale = ref["preds"].abs().max().item()
    dp = (ours["preds"] - ref["preds"]).abs().amax(dim=(0, 2, 3)) / scale      # per emitted frame
    for k, v in enumerate(dp.tolist()):
        assert v < tol(k), f"{what}: rollout predictions differ at frame {k}: {dp.tolist()}"
    n = len(ours["test_losses"])
    for i, (a, b) in enumerate(zip(ours["test_losses"], ref["test_losses"])):
        assert _rel(a, b) < max(1e-3, 10 * tol(i * F // n)), f"{what}: test MSE of frame {i}: {a} vs {b}"
    es = ref["energies"].abs().max().item()
    de = (ours["energies"] - ref["energies"]).abs().amax(dim=(0, 2)) / es
    for k, v in enumerate(de.tolist()):
        assert v < max(1e-3, 10 * tol(k * F // len(de))), f"{what}: energy curves differ: {de.tolist()}"
    assert _rel(ours["test_loss"], ref["test_loss"]) < max(1e-2, 10 * tol(F - 1))


class _OracleEGNO(torch.nn.Module):
    """The oracle restatement behind the reference's module interface (parameters borrowed from a reference module)."""

    def __init__(self, holder, T, L):
        super().__init__()
        self.holder, self.num_timesteps, self.L = holder, T, L

    def forward(self, x, h, edge_index, edge_fea, v=None, loc_mean=None, timesteps_in=None, timesteps_out=None):
        p = dict(self.holder.named_parameters())
        return O.egno_forward(p, x, h, edge_index[0], edge_index[1], edge_fea, v, loc_mean, timesteps_out,
                              n_layers=self.L, num_timesteps=self.num_timesteps)


class _OracleSEGNO(torch.nn.Module):
    def __init__(self, holder):
        super().__init__()
        self.holder = holder

    def forward(self, his, x, edges, v, edge_attr, T=10, in_steps=None):
        p = dict(self.holder.named_parameters())
        return O.segno_forward(p, his, x, edges[0], edges[1], v, edge_attr, T=T, recurrent=True)


@pytest.fixture(scope="module")
def ref():
    R = RL.load_reference_drivers()
    R.SEGNO.forward = RL.segno_intended_forward      # SURVEY.md §0 defect 1: HEAD's forward returns its inputs
    return R


# ------------------------------------------------------------------------------------------------ CPU tier
@needs_ref
def test_oracle_restatement_through_the_reference_drivers(ref, tmp_path):
    """not gpu: pins the oracle at driver level (training dynamics, rollout, energies), and proves the harness."""
    d = DF.write_dataset(tmp_path / "c", "charged", 5, {"train": 16, "valid": 8, "test": 8}, length=6000, seed=43)
    torch.manual_seed(1)
    m_ref = ref.EGNO(num_timesteps=8, device="cpu", **EGNO_KW)
    torch.manual_seed(1)
    holder = ref.EGNO(num_timesteps=8, device="cpu", **EGNO_KW)
    a = H.egno_driver_run(ref, _OracleEGNO(holder, 8, 4), "cpu", d, 5, 8, 8, 2, 3)
    b = H.egno_driver_run(ref, m_ref, "cpu", d, 5, 8, 8, 2, 3)
    _compare(a, b, "oracle EGNO", per_call=8)
    g = DF.write_dataset(tmp_path / "g", "gravity", 5, {"train": 16, "valid": 8, "test": 8}, length=4000, seed=47)
    torch.manual_seed(1)
    s_ref = ref.SEGNO(device="cpu", **SEGNO_KW)
    torch.manual_seed(1)
    s_holder = ref.SEGNO(device="cpu", **SEGNO_KW)
    a = H.segno_driver_run(ref, _OracleSEGNO(s_holder), "cpu", g, 5, 10, 8, 2, 3)
    b = H.segno_driver_run(ref, s_ref, "cpu", g, 5, 10, 8, 2, 3)
    _compare(a, b, "oracle SEGNO")


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@needs_ref
@pytest.mark.parametrize("n_balls,T,traj_len,length", [(5, 8, 4, 8000), (20, 10, 3, 8000)])
def test_reference_egno_drivers_run_the_cuda_module(ref, tmp_path, n_balls, T, traj_len, length):
    import no_node_comparison_b200 as nb

    dev = torch.device("cuda:0")
    d = DF.write_dataset(tmp_path / "c", "charged", n_balls, {"train": 32, "valid": 16, "test": 16}, length=length, seed=43,
                         device=dev)
    torch.manual_seed(1)
    m_ref = ref.EGNO(num_timesteps=T, device="cpu", **EGNO_KW)
    m = nb.EGNO(num_timesteps=T, device=dev, **EGNO_KW)
    m.load_state_dict(m_ref.state_dict())
    ours = H.egno_driver_run(ref, m, dev, d, n_balls, T, 16, 2, traj_len)
    theirs = H.egno_driver_run(ref, m_ref, "cpu", d, n_balls, T, 16, 2, traj_len)
    _compare(ours, theirs, f"EGNO N={n_balls}", per_call=T)


@pytest.mark.gpu
@needs_ref
@pytest.mark.parametrize("kind,n_balls,traj_len,length", [("gravity", 5, 5, 6000), ("gravity", 20, 4, 5000), ("charged", 5, 3, 8000)])
def test_reference_segno_drivers_run_the_cuda_module(ref, tmp_path, kind, n_balls, traj_len, length):
    import no_node_comparison_b200 as nb

    dev = torch.device("cuda:0")
    d = DF.write_dataset(tmp_path / "g", kind, n_balls, {"train": 32, "valid": 16, "test": 16}, length=length, seed=47,
                         device=dev)
    torch.manual_seed(1)
    s_ref = ref.SEGNO(device="cpu", **SEGNO_KW)
    s = nb.SEGNO(device=dev, **SEGNO_KW)
    s.load_state_dict(s_ref.state_dict())
    ours = H.segno_driver_run(ref, s, dev, d, n_balls, 10, 16, 2, traj_len, dataset=kind)
    theirs = H.segno_driver_run(ref, s_ref, "cpu", d, n_balls, 10, 16, 2, traj_len, dataset=kind)
    _compare(ours, theirs, f"SEGNO {kind} N={n_balls}")
