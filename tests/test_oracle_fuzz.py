"""Differential fuzzing of the CPU restatement against the reference's own C++: random and adversarial pairs through
raw_align / al2subs / compute_lambda with varying scores, bands and modes; end-to-end runs on small random inputs with
random options.  The reference's answers for these seeded cases are stored under tests/golden/ (fuzz_pairs.npz,
e2e_fuzz<i>.npz; tools/make_golden_fuzz.py regenerates them from the compiled reference)."""
import os

import numpy as np

from oracle import port
from tests import cases

N_E2E = 6


def _rseq(rng, n):
    return "".join("ACGT"[c] for c in rng.integers(0, 4, size=n))


def _mut(rng, s, nsub, nindel):
    s = list(s)
    for _ in range(nsub):
        p = int(rng.integers(0, len(s)))
        s[p] = "ACGT"[("ACGT".index(s[p]) + int(rng.integers(1, 4))) % 4]
    for _ in range(nindel):
        p = int(rng.integers(1, len(s) - 1))
        n = int(rng.integers(1, 4))
        if rng.random() < 0.5:
            del s[p:p + n]
        else:
            s[p:p] = [s[p]] * n if rng.random() < 0.5 else list(_rseq(rng, n))
    return "".join(s)


def pair_cases():
    """The seeded pair corpus: -> list of (it, a, qa, b, qb, pair options)."""
    rng = np.random.default_rng(77)
    out = []
    for it in range(400):
        L = int(rng.integers(12, 140))
        a = _rseq(rng, L) if rng.random() < 0.8 else (_rseq(rng, int(rng.integers(1, 4))) * L)[:L]
        b = _mut(rng, a, int(rng.integers(0, 10)), int(rng.integers(0, 3))) if rng.random() < 0.85 else _rseq(rng, L + int(rng.integers(-4, 5)))
        if len(b) < 8:
            continue
        qa = rng.integers(0, 41, size=len(a)).astype(np.uint8)
        qb = rng.integers(0, 41, size=len(b)).astype(np.uint8)
        mode = int(rng.integers(0, 3))
        o = dict(match=int(rng.integers(1, 7)), mismatch=-int(rng.integers(1, 7)), gap=-int(rng.integers(1, 10)),
                 band_size=int(rng.choice([-1, 0, 1, 2, 3, 5, 8, 16, 17, 32])), gapless=bool(rng.random() < 0.8),
                 SSE=int(rng.choice([0, 1, 2])))
        if mode == 0:
            o.update(vectorized_alignment=True, homo_gap=o["gap"])
        elif mode == 1:
            o.update(vectorized_alignment=False, homo_gap=o["gap"])
        else:
            o.update(vectorized_alignment=False, homo_gap=-int(rng.integers(0, 5)))
        kd = float(rng.choice([0.42, 1.0, 0.2]))
        use_k = bool(rng.random() < 0.85)
        out.append((it, a, qa, b, qb, dict(o, use_kmers=use_k, kdist_cutoff=kd)))
    return out


def e2e_cases():
    """The seeded end-to-end inputs: -> list of (seqs, abundances, priors, quals, dada_uniques options)."""
    from tools import synth
    rng = np.random.default_rng(99)
    out = []
    for it in range(N_E2E):
        seqs, ab, q, _ = synth.illumina(int(rng.integers(150, 500)), L=int(rng.choice([60, 100, 150])), nvar=int(rng.integers(3, 20)),
                                        max_subs=int(rng.integers(3, 30)), seed=1000 + it, lowq_frac=float(rng.choice([0.002, 0.02])))
        o = dict(band_size=int(rng.choice([4, 16, 32])), omegaA=float(rng.choice([1e-40, 1e-10, 1e-4])),
                 greedy=bool(rng.random() < 0.7), gapless=bool(rng.random() < 0.7), use_kmers=bool(rng.random() < 0.8),
                 kdist_cutoff=float(rng.choice([0.42, 0.3])), min_fold=float(rng.choice([1.0, 1.5])),
                 min_hamming=int(rng.choice([1, 2])), min_abund=int(rng.choice([1, 2])),
                 detect_singletons=bool(rng.random() < 0.3), omegaC=float(rng.choice([1e-40, 1e-5])), homo_gap=-8)
        pri = (rng.random(len(seqs)) < 0.1).astype(np.uint8) if rng.random() < 0.5 else None
        out.append((seqs, ab, pri, q, o))
    return out


# per-pair vectors stored concatenated in fuzz_pairs.npz: map has len(a) entries, the others max(nsubs, 0)
PAIR_VECTORS = ("map", "pos", "nt0", "nt1", "q0", "q1")


def golden_pairs():
    """-> {it: reference result of pair_cases()' pair `it`} from tests/golden/fuzz_pairs.npz."""
    z = np.load(os.path.join(cases.GOLDEN, "fuzz_pairs.npz"), allow_pickle=False)
    vec = {}
    for k in PAIR_VECTORS:
        n = z["map_len"] if k == "map" else np.maximum(z["nsubs"], 0)
        vec[k] = np.split(z[k], np.cumsum(n)[:-1])
    out = {}
    for i, it in enumerate(z["it"].tolist()):
        r = dict(shrouded=bool(z["shrouded"][i]), lam=float(z["lam"][i]), nsubs=int(z["nsubs"][i]),
                 al0=str(z["al0"][i]), al1=str(z["al1"][i]))
        r.update({k: vec[k][i] for k in PAIR_VECTORS})
        r["nt0"], r["nt1"] = r["nt0"].tobytes(), r["nt1"].tobytes()
        out[it] = r
    return out


def test_pair_level_fuzz():
    err = cases.tperr1()
    want = golden_pairs()
    n_nw = 0
    todo = pair_cases()
    assert sorted(want) == [c[0] for c in todo]
    for it, a, qa, b, qb, o in todo:
        p = port.pair(a, qa, b, qb, err, **o)
        r = want[it]
        assert p["shrouded"] == r["shrouded"], (it, o)
        if r["shrouded"]:
            assert p["lam"] == 0.0 == r["lam"]
            continue
        assert (p["al0"], p["al1"]) == (r["al0"], r["al1"]), (it, o, a, b)
        assert p["nsubs"] == r["nsubs"] and p["lam"] == r["lam"], (it, o)
        assert np.array_equal(p["map"], r["map"]) and np.array_equal(p["pos"], r["pos"])
        assert p["nt0"] == r["nt0"] and p["nt1"] == r["nt1"]
        assert np.array_equal(p["q0"], r["q0"]) and np.array_equal(p["q1"], r["q1"])
        n_nw += p["kind"] == 2
    assert n_nw > 150


def test_end_to_end_fuzz_random_options():
    from tests.test_oracle import load_golden
    err = cases.tperr1()
    for it, (seqs, ab, pri, q, o) in enumerate(e2e_cases()):
        a = port.dada_uniques(seqs, ab, pri, err, q, **o)
        b = load_golden("fuzz%d" % it)
        pb = None
        if pri is not None:
            pb = np.ones(len(b["clustering"]["sequence"]), dtype=bool)     # birth_from of prior-born clusters is undefined in the reference
        cases.assert_same(a, b, rtol=1e-15, prior_born=pb, label="fuzz%d %s" % (it, o))
