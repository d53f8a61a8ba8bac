"""oracle/ — TEST INFRASTRUCTURE, not product code.

A CPU restatement (plain PyTorch, CPU tensors) of the reference's EGNO / SEGNO
hot path, used only as the *checker*:

  * ``tests/``                      – parity tests compare the CUDA path with it
  * ``__graft_entry__.smoke()``     – one tiny check on cuda:0
  * ``bench.py``                    – the ``cpu_baseline`` leg and ``--impl reference``

Nothing in ``no-node-comparison_b200/`` imports this package; the product path
fails loudly when its CUDA extension is missing.

Parity pin status: the reference ships NO tests, golden vectors or known-answer
fixtures for this path (SURVEY.md §4, §8c) -> "parity unpinned by reference
tests".  The oracle is instead pinned against outputs of the reference's own
modules: ``tests/golden/make_golden.py`` imports the reference
(through ``oracle/ref_loader.py``), runs the real
``EGNO`` / ``SEGNO.forward_step`` on seeded inputs and commits inputs, weights,
outputs and parameter gradients under ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` checks the restatement in ``nbody_oracle.py``
against those vectors on every run.
"""
