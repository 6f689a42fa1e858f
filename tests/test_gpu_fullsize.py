"""BASELINE-size checks on the GPU (configs[1]: 1e5 synthetic 250-nt uniques): size-independent properties
(tests/properties.py, pinned on the oracle at small sizes), run-to-run determinism, one-shot == resident, and the output
against the reference's own C++ on the same input (tests/golden/e2e_fullsize_1e5.npz, tools/make_golden_fuzz.py: every
per-cluster field whole, the per-unique map / pval at a seeded sample).  bench.py diffs the 1e6 workload against the same library in its cpu_baseline leg."""
import numpy as np
import pytest

from tests import cases
from tests.properties import check_invariants

pytestmark = pytest.mark.gpu


def test_1e5_uniques_invariants_determinism_and_paths_agree():
    import dada2_b200
    from tools import synth
    seqs, ab, q, truth = synth.illumina(100000, seed=12345)
    err = cases.tperr1()
    res = dada2_b200.Resident(seqs, ab, None, q)
    a = res.run(err)
    b = res.run(err)
    res.close()
    c = dada2_b200.dada_uniques(seqs, ab, None, err, q)          # one-shot C-ABI path
    cases.assert_same(b, a, rtol=0.0, label="rerun")
    cases.assert_same(c, a, rtol=0.0, label="one-shot vs resident")
    check_invariants(seqs, ab, a)
    found = set(a["clustering"]["sequence"])
    assert len(found) == 100 and sum(v in found for v in truth["variants"]) >= 95     # the planted variants are recovered
    from tests.test_oracle import load_golden
    want = load_golden("fullsize_1e5")                            # the reference's C++ on the same 1e5 uniques
    idx = want.pop("sample_idx")
    cases.assert_same(dict(a, map=np.asarray(a["map"])[idx], pval=np.asarray(a["pval"])[idx]), want, rtol=1e-10,
                      label="1e5 uniques vs the reference's C++ (map / pval at %d sampled uniques)" % len(idx))
    st = a["stats"]
    assert st["gpu_launches"] > 1000 and st["n_nw"] > 1_000_000 and st["n_final_nw"] == 100000
