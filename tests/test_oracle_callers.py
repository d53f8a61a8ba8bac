"""The oracle's restatements of the CALLERS' helpers against the reference's own functions (VERDICT r01 weak / 3e):

  oracle.egno_features / egno_features_multi  vs  prepare_inputs            EGNO/main_simulation_simple_no.py:311-339
  oracle.energy_charged / energy_gravity      vs  utils.conserved_energy_fun utils.py:126-219
  oracle.trajectory_mse                       vs  the loss lines of run_epoch main_simulation_simple_no.py:268-276

The reference is imported through oracle/ref_loader.py (the original checkout, or the unmodified copy under oracle/_ref
made by oracle/make_ref.py); the tests that call it skip without it.  The loss lines are written out in the test itself
and need no reference."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import nbody_oracle as O
from oracle import ref_loader as RL
from tests.helpers import rel_err

needs_ref = pytest.mark.skipif(not RL.reference_available(), reason="reference not installed (run oracle/make_ref.py)")


@pytest.fixture(scope="module")
def ref():
    return RL.load_reference_drivers()


def _state(B, N, seed, frames=None):
    g = torch.Generator().manual_seed(seed)
    lead = (B, N) if frames is None else (B, frames, N)
    loc = torch.randn(*lead, 3, generator=g) * 1.3
    vel = torch.randn(*lead, 3, generator=g) * 0.4
    q = (torch.randint(0, 2, (B, N, 1), generator=g).float() * 2 - 1)
    return loc, vel, q


@needs_ref
@pytest.mark.parametrize("B,N", [(3, 5), (2, 20)])
def test_egno_features_match_prepare_inputs(ref, B, N):
    loc, vel, q = _state(B, N, 10 * B + N)
    row, col = O.canonical_edges(B, N)
    qq = (q.reshape(-1, 1)[row] * q.reshape(-1, 1)[col])                       # dataset_simple.py:52-53
    r_loc, r_vel, r_ea, r_nodes, r_mean = ref.egno_main.prepare_inputs(loc, vel, qq, (row, col), N, 1, charges=q)
    x, v, ea, nodes, mean = O.egno_features(loc, vel, q, row, col)
    for a, b in ((x, r_loc), (v, r_vel), (ea, r_ea), (nodes, r_nodes), (mean, r_mean)):
        assert a.shape == b.shape and torch.equal(a, b)


@needs_ref
def test_egno_multi_input_features_match_prepare_inputs(ref):
    B, N, nin = 3, 5, 3
    loc, vel, q = _state(B, N, 7, frames=nin)                                    # loader layout [B, num_inputs, N, 3]
    row, col = O.canonical_edges(B, N)
    qq = (q.reshape(-1, 1)[row] * q.reshape(-1, 1)[col])
    r_loc, r_vel, r_ea, r_nodes, r_mean = ref.egno_main.prepare_inputs(loc, vel, qq, (row, col), N, nin, charges=q)
    x, v, ea, nodes, mean = O.egno_features_multi(loc.transpose(0, 1), vel.transpose(0, 1), q, row, col)
    for a, b in ((x, r_loc), (v, r_vel), (ea, r_ea), (nodes, r_nodes), (mean, r_mean)):
        assert a.shape == b.shape and rel_err(a, b) < 1e-7


@needs_ref
@pytest.mark.parametrize("kind", ["charged", "gravity"])
def test_energies_match_conserved_energy_fun(ref, kind):
    B, N = 6, 20
    loc, vel, q = _state(B, N, 3)
    if kind == "gravity":
        q = q.abs() * torch.rand(B, N, 1, generator=torch.Generator().manual_seed(1)) + 0.5     # masses
    batch = torch.arange(B).repeat_interleave(N)
    want = ref.utils.conserved_energy_fun(kind, loc.reshape(-1, 3), vel.reshape(-1, 3), q.reshape(-1, 1), batch=batch)
    got = (O.energy_charged if kind == "charged" else O.energy_gravity)(loc, vel, q)
    assert np.asarray(want).shape == (B,)
    assert rel_err(got, torch.as_tensor(np.asarray(want), dtype=torch.float32)) < 2e-6


@pytest.mark.parametrize("only_first", [False, True])
def test_trajectory_mse_matches_the_loss_lines_of_run_epoch(only_first):
    """main_simulation_simple_no.py:268-276 written out with the reference's own criterion object."""
    T, B, N = 4, 3, 5
    g = torch.Generator().manual_seed(2)
    pred = torch.randn(T * B * N, 3, generator=g)
    tgt = torch.randn(B * N, T, 3, generator=g)
    crit = torch.nn.MSELoss(reduction="none")
    losses = crit(pred.view(T, B * N, 3).transpose(0, 1).contiguous().view(-1, 3), tgt.reshape(-1, 3)).view(B * N, T, 3)
    losses = torch.mean(losses, dim=(0, 2))
    want = losses[0] if only_first else torch.mean(losses)
    loss, per_frame = O.trajectory_mse(pred, tgt, only_first)
    assert rel_err(per_frame, losses) < 1e-6 and abs(float(loss) - float(want)) < 1e-6 * abs(float(want))   # summation order
