"""Distance MLE between contig pairs (SURVEY.md §8(f) rank 4; gt_scaffolder_bamparser.c:385-598).

The oracle is the reference's own estimate_dist_using_mle: oracle/ref_bam_driver.c includes
gt_scaffolder_bamparser.c unmodified and calls its static functions.

CPU: the host build of gtsb_mle_host (tests/emul/mle_emul.cpp: the same preparation, stage function,
     ranking rule and decision, the device scan as loops) against the reference on random
     libraries -- forward-reverse and reverse-forward, unimodal and flat distributions, ranges cut
     by the distribution and by min/max distance, fragments outside the distribution, repeated
     fragment sizes, single fragments, ties; the ranking filter must never change the answer
     (keep_all run) and must keep only a few thetas.
GPU: gtsb_mle_host against the same host build, and through it against the reference.
"""
import numpy as np
import pytest

import oracle_lib as O
import parse_emul as PE

needs_ref = pytest.mark.skipif(not O.have_refbam(), reason="compiled reference estimator (oracle/_ref) not available")


@pytest.fixture(scope="module", autouse=True)
def _built():
    O.build_oracles()


def make_pmf(rng, kind, nof):
    x = np.arange(nof, dtype=np.float64)
    if kind == "normal":
        mu, sd = nof * rng.uniform(0.3, 0.6), nof * rng.uniform(0.03, 0.12)
        h = np.exp(-0.5 * ((x - mu) / sd) ** 2)
    elif kind == "bimodal":
        h = np.exp(-0.5 * ((x - nof * 0.3) / (nof * 0.04)) ** 2) + 0.6 * np.exp(-0.5 * ((x - nof * 0.7) / (nof * 0.06)) ** 2)
    elif kind == "flat":
        h = np.ones(nof)
    else:                                  # ragged histogram with empty bins
        h = rng.integers(0, 40, nof).astype(np.float64) * (rng.random(nof) < 0.7)
    h = h / h.sum()
    minp = float(rng.choice([1e-12, 1.0 / (50 * nof), 1e-6]))
    pmf = np.where(h > minp, h, minp)      # create_pmf floors at minp (bamparser.c:367-383)
    return pmf, minp


def make_pairs(rng, pmf, n_pairs, rf, ma):
    nof = len(pmf)
    cdf = np.cumsum(pmf / pmf.sum())
    pairs = []
    for _ in range(n_pairs):
        n = int(rng.choice([1, 2, 3, 8, 30, 120]))
        true_gap = int(rng.integers(-40, nof // 2))
        sizes = np.searchsorted(cdf, rng.random(n)).astype(np.int64) - true_gap        # provisional sizes
        if rng.random() < 0.3:
            sizes[rng.integers(0, n)] += int(rng.integers(-nof, 2 * nof))              # an outlier
        if rng.random() < 0.4 and n > 2:
            sizes[1] = sizes[0]                                                        # a repeated size
        if not rf:
            sizes = np.maximum(sizes, 2 * (ma - 1) + rng.integers(0, 3, n))
        start = rng.integers(0, 5000, n).astype(np.int64)
        frag = np.stack([start, start + sizes], axis=1)
        pairs.append((frag, ma, int(rng.integers(ma + 200, 30000)), int(rng.integers(ma + 200, 30000))))
    return pairs


CASES = [(kind, rf, seed) for seed, kind in enumerate(["normal", "bimodal", "flat", "ragged"]) for rf in (False, True)]


@needs_ref
@pytest.mark.parametrize("kind,rf,seed", CASES)
def test_host_build_equals_the_reference(kind, rf, seed):
    rng = np.random.default_rng(700 + seed * 2 + int(rf))
    nof = int(rng.choice([60, 300, 900]))
    pmf, minp = make_pmf(rng, kind, nof)
    ma = int(rng.choice([1, 30, 100]))
    pairs = make_pairs(rng, pmf, 25, rf, ma)
    for min_dist, max_dist in ((-99, 100000), (-20, 150), (0, 40), (50, 10)):
        got = PE.mle(pairs, pmf, minp, rf, min_dist, max_dist)
        everything = PE.mle(pairs, pmf, minp, rf, min_dist, max_dist, keep_all=True)
        assert got is not None and everything is not None
        for i, (frag, m, lr, lm) in enumerate(pairs):
            exp = O.ref_estimate_dist(frag, m, lr, lm, pmf, minp, rf, min_dist, max_dist)
            assert (int(got[0][i]), int(got[1][i])) == exp, (kind, rf, min_dist, max_dist, i)
            assert (int(everything[0][i]), int(everything[1][i])) == exp
        if kind in ("normal", "bimodal") and got[2] > 5000:
            assert got[3] * 20 < got[2], "the ranking keeps too many thetas: %d of %d" % (got[3], got[2])


def test_negative_probability_is_refused():
    pmf = np.array([0.2, 0.5, -0.1, 0.4])
    frag = np.array([[0, 2]], np.int64)
    assert PE.mle([(frag, 1, 500, 600)], pmf, 1e-6, True, -5, 5) is None


# ------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("kind,rf,seed", CASES)
def test_device_equals_host_build(pkg, kind, rf, seed):
    rng = np.random.default_rng(900 + seed * 2 + int(rf))
    nof = int(rng.choice([300, 900]))
    pmf, minp = make_pmf(rng, kind, nof)
    ma = int(rng.choice([1, 30, 100]))
    pairs = make_pairs(rng, pmf, 200, rf, ma)
    g = pkg.ScaffoldGraphB200()
    for min_dist, max_dist in ((-99, 100000), (-20, 150), (50, 10)):
        exp = PE.mle(pairs, pmf, minp, rf, min_dist, max_dist)
        dist, used = g.mle(*PE.mle_arrays(pairs), pmf, minp, rf, min_dist, max_dist)
        assert np.array_equal(dist, exp[0]) and np.array_equal(used, exp[1])
    if O.have_refbam():
        for i in range(0, len(pairs), 17):
            frag, m, lr, lm = pairs[i]
            assert (int(dist[i]), int(used[i])) == O.ref_estimate_dist(frag, m, lr, lm, pmf, minp, rf, 50, 10)
    with pytest.raises(RuntimeError, match="negative probability"):
        g.mle(*PE.mle_arrays(pairs[:1]), np.array([0.5, -0.5]), 1e-6, rf, -5, 5)
    g.close()


@pytest.mark.gpu
def test_device_mle_at_size(pkg):
    import json
    import os
    rng = np.random.default_rng(12)
    pmf, minp = make_pmf(rng, "normal", 1000)
    pairs = make_pairs(rng, pmf, 20000, True, 1)
    g = pkg.ScaffoldGraphB200()
    a = PE.mle_arrays(pairs)
    g.mle(*a, pmf, minp, True, -99, 100000)
    g.set_profile(True)
    dist, used = g.mle(*a, pmf, minp, True, -99, 100000)
    prof = {k: round(v[0], 4) for k, v in g.profile().items()}
    exp = PE.mle(pairs[:300], pmf, minp, True, -99, 100000)
    assert np.array_equal(dist[:300], exp[0]) and np.array_equal(used[:300], exp[1])
    report = dict(contig_pairs=len(pairs), fragments=int(a[0][-1]), pmf_nof=len(pmf), kernel_ms=prof)
    print("\n[mle]", json.dumps(report))
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "mle_profile.json"), "w") as f:
            json.dump(report, f, indent=1)
    g.close()
