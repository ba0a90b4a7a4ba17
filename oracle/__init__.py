"""oracle/ -- TEST INFRASTRUCTURE ONLY.

CPU restatement of the reference's embedding-to-distance path
(KevinWangHP/Anomaly-Clustering).  Nothing in the product package
(`anomaly_clustering_b200/`) may import from here; only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs do, and there only as the checker / the reported CPU baseline.

Parity status
-------------
* stages 1-3 (Z, w, alpha, X): the reference has NO golden vectors or
  known-answer tests for this path (SURVEY.md section 8c).  The restatement is
  pinned by executing the reference's own Python code (imported from the
  checkout AC_REFERENCE_DIR names by `oracle/ref_import.py`) on seeded
  synthetic inputs; `oracle/make_golden.py` stores those reference outputs as
  fixtures in `tests/golden/` and `tests/test_oracle_golden.py` re-checks the
  restatement against them on every run.
* stage "X -> Ward -> NMI/ARI/F1": pinned by the reference's shipped result
  artefacts (alpha/X pickles + tau_result.csv); a compact extract is committed
  in `tests/golden/shipped_cluster_golden.npz`.
* the arithmetic itself lives in PyTorch (reference pins torch==1.12.1; this
  image has 2.11) -- parity at the torch boundary is pinned only by executing
  this image's torch.
"""
