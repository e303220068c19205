"""CPU oracle for the D4PG learner hot path -- TEST INFRASTRUCTURE ONLY.

Nothing in the product package (`d4pg-pytorch_b200/`) may import this package.
Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s `cpu_baseline` /
`--impl reference` legs use it, and only as the checker / the CPU arm.

Parity status: PINNED.  The reference has no tests or golden vectors of its own
(SURVEY.md section 4), so the pin is the reference code itself, imported unmodified
from /root/reference behind the 4-item compat shim in `oracle/ref_shim.py` and
run in the build container:
  * `tests/golden/make_golden.py` dumps reference outputs to `tests/golden/*.npz`
    (NumPy 2.3.5 / torch 2.11.0 CPU dtype semantics, see SURVEY.md H11);
  * `tests/test_oracle_golden.py` and `tests/test_oracle_vs_reference.py` check
    the oracle against the committed fixtures everywhere.
"""
