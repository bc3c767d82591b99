"""oracle/ -- CPU restatement of the reference hot path.  TEST INFRASTRUCTURE ONLY.

May be imported only from tests/, __graft_entry__.smoke() / build() and bench.py's cpu_baseline /
--impl reference legs.  Never from opentransformer_b200 (the product).

Pinning: (1) committed fixtures produced by the real reference (tests/golden/, tests/test_oracle_golden.py);
(2) oracle/_ref/ -- the reference's own Python modules byte-compiled by oracle/build_ref.py (git-ignored):
tests/golden/make_reference_checks.py records from it what the reference computes for tests/test_oracle_ref.py, and
bench.py's reference arm times the reference itself (cpu_baseline.kind "reference"; "port" only when _ref is absent).
"""
