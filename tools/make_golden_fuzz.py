"""Generates the goldens of the differential tests from the REFERENCE's own C++ (oracle/_ref/libdada2ref.so, compiled
unmodified by `make -C oracle ref`; needs the reference sources):
    fuzz_pairs.npz          sub_new + compute_lambda_ts for tests/test_oracle_fuzz.py's pair_cases()
    e2e_fuzz<i>.npz         dada_uniques for tests/test_oracle_fuzz.py's e2e_cases()
    bimera_fuzz.npz         C_table_bimera2 and the pair primitives for tests/test_bimera_oracle.py's fuzz_cases()
    e2e_fullsize_1e5.npz    dada_uniques on tests/test_gpu_fullsize.py's 1e5 uniques; the per-unique `map` and `pval`
                            at FULLSIZE_SAMPLE seeded positions (`sample_idx`), every other field whole
Run:  python tools/make_golden_fuzz.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref                  # noqa: E402
from tests import cases                 # noqa: E402
from tools.make_golden import save_res  # noqa: E402

G = cases.GOLDEN
FULLSIZE_SAMPLE = 8192


def pairs():
    from tests.test_oracle_fuzz import PAIR_VECTORS, pair_cases
    err = cases.tperr1()
    rec = {k: [] for k in ("it", "shrouded", "lam", "nsubs", "al0", "al1", "map_len") + PAIR_VECTORS}
    for it, a, qa, b, qb, o in pair_cases():
        r = ref.pair(a, qa, b, qb, err, **o)
        rec["it"].append(it)
        rec["map_len"].append(len(r["map"]))
        for k in ("shrouded", "lam", "nsubs", "al0", "al1"):
            rec[k].append(r[k])
        for k in PAIR_VECTORS:
            rec[k].append(np.frombuffer(r[k], np.uint8) if isinstance(r[k], bytes) else r[k])
    out = {k: np.array(v) for k, v in rec.items() if k not in PAIR_VECTORS}
    out.update({k: np.concatenate(rec[k]) for k in PAIR_VECTORS})
    np.savez_compressed(os.path.join(G, "fuzz_pairs.npz"), **out)
    print("fuzz pairs", len(rec["it"]))


def e2e():
    from tests.test_oracle_fuzz import e2e_cases
    err = cases.tperr1()
    for it, (seqs, ab, pri, q, o) in enumerate(e2e_cases()):
        res = ref.dada_uniques(seqs, ab, pri, err, q, **o)
        save_res(os.path.join(G, "e2e_fuzz%d.npz" % it), res)
        print("e2e fuzz", it, len(seqs), "uniques ->", len(res["clustering"]["sequence"]))


def bimera():
    from tests.test_bimera_oracle import FUZZ_PAIR_INTS, fuzz_cases
    out = {}
    for n, (seqs, mat, o, prs) in enumerate(fuzz_cases()):
        out["t%d__nflag" % n], out["t%d__nsam" % n] = ref.table_bimera(mat, seqs, **o)
        rs = [ref.bimera_pair(seqs[j], seqs[k], **{x: o[x] for x in ("allow_one_off", "max_shift")}) for j, k in prs]
        out["t%d__pair_ints" % n] = np.array([[r[x] for x in FUZZ_PAIR_INTS] for r in rs], np.int32)
        out["t%d__al0" % n] = np.array([r["al0"] for r in rs])
        out["t%d__al1" % n] = np.array([r["al1"] for r in rs])
    np.savez_compressed(os.path.join(G, "bimera_fuzz.npz"), **out)
    print("bimera fuzz", n + 1, "tables")


def fullsize():
    from tools import synth
    seqs, ab, q, _ = synth.illumina(100000, seed=12345)
    ref.set_threads(os.cpu_count() or 1)
    res = ref.dada_uniques(seqs, ab, None, cases.tperr1(), q, multithread=True)
    idx = np.sort(np.random.default_rng(1).choice(len(seqs), FULLSIZE_SAMPLE, replace=False)).astype(np.int32)
    res["map"], res["pval"] = res["map"][idx], res["pval"][idx]
    res["sample_idx"] = idx
    save_res(os.path.join(G, "e2e_fullsize_1e5.npz"), res)
    print("fullsize 1e5 ->", len(res["clustering"]["sequence"]), "partitions")


if __name__ == "__main__":
    pairs()
    e2e()
    bimera()
    fullsize()
