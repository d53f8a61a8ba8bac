#!/usr/bin/env python
"""Golden trajectories of the reference's simulators (imports the reference's synthetic_sim.py via oracle/ref_loader.py).

For every case: seed the global numpy stream, draw the initial conditions with oracle.sim_oracle's samplers (which
mirror the reference's draw order), re-seed, run the reference's own sample_trajectory -> the stored frames belong to
exactly those initial conditions.  Writes tests/golden/sim_<case>.npz (float64).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_loader, sim_oracle as S  # noqa: E402

ref_loader._install_stubs()
sys.path.insert(0, ref_loader.REFERENCE_ROOT)
import synthetic_sim  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [("charged", 5, 2000, 100, 43), ("charged", 20, 1000, 100, 44), ("gravity", 5, 1000, 100, 45), ("gravity", 20, 600, 100, 46)]

for kind, n, T, sf, seed in CASES:
    ntraj = 2
    if kind == "charged":
        np.random.seed(seed)
        ics = [S.charged_initial_conditions(n, T // sf - 1) for _ in range(ntraj)]
        np.random.seed(seed)
        sim = synthetic_sim.ChargedParticlesSim(noise_var=0.0, n_balls=n, vel_norm=0.5)
        outs = [sim.sample_trajectory(T=T, sample_freq=sf) for _ in range(ntraj)]
        for (l0, v0, q), (loc, vel, edges, charges) in zip(ics, outs):
            assert np.array_equal(q, charges), "initial-condition sampler out of step with the reference"
        np.savez_compressed(os.path.join(HERE, f"sim_{kind}_n{n}.npz"), T=T, sample_freq=sf,
                            loc0=np.stack([i[0] for i in ics]), vel0=np.stack([i[1] for i in ics]),
                            charges=np.stack([i[2] for i in ics]), loc=np.stack([o[0] for o in outs]),
                            vel=np.stack([o[1] for o in outs]))
    else:
        np.random.seed(seed)
        ics = [S.gravity_initial_conditions(n, T // sf) for _ in range(ntraj)]
        np.random.seed(seed)
        sim = synthetic_sim.GravitySim(noise_var=0.0, n_balls=n)
        outs = [sim.sample_trajectory(T=T, sample_freq=sf) for _ in range(ntraj)]
        for (p0, v0, m), (pos, vel, force, mass) in zip(ics, outs):
            assert np.array_equal(m, mass), "initial-condition sampler out of step with the reference"
        np.savez_compressed(os.path.join(HERE, f"sim_{kind}_n{n}.npz"), T=T, sample_freq=sf,
                            pos0=np.stack([i[0] for i in ics]), vel0=np.stack([i[1] for i in ics]),
                            mass=np.stack([i[2] for i in ics]), pos=np.stack([o[0] for o in outs]),
                            vel=np.stack([o[1] for o in outs]), force=np.stack([o[2] for o in outs]))
    print("wrote", kind, n)
