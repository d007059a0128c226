"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the dense-correspondence matching path.

Nothing under oracle/ is imported by the product (midvision-probe_b200/).  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it, and only as the
checker or the timed CPU baseline.

Parity status: PINNED against the reference itself run here (the second route of the oracle rule): the
reference ships no tests, golden vectors or known-answer files for this path, so
  * oracle/reference_loader.py imports the reference's own, unmodified evals/utils/correspondence.py and
    evaluate_spair_correspondence.py from a checkout of the reference project (oracle/_ref/ or
    $MV_REFERENCE_ROOT; stand-ins only for modules that are not installed:
    hydra / omegaconf, and the four faiss symbols);
  * oracle/make_golden.py runs them on seeded inputs and commits the outputs under tests/golden/ (the
    reference is not part of this repository);
  * oracle/restated.py -- the restatement used everywhere else -- is checked against both (tests/test_oracle.py; the comparisons
    with the reference itself run only where a checkout of it is present).
The one restated third-party piece is faiss-gpu 1.8.0's GpuIndexFlatL2.search (README.md:60; call sites
evals/utils/correspondence.py:11, :20-22; not part of the reference tree and not installed for these tests): its published
contract -- exact L2 top-k, ascending, int64 labels -- is what oracle/faiss_shim.py implements; the reference
discards its distances (:50), so only the order of fp32-rounding-level ties can differ from the real library.
"""
