"""CPU: the oracle's restatement of DenseMatcher::match against the REAL reference matcher -- okvis_matcher's own sources
compiled unmodified (oracle/Makefile.ref; the one part of the reference that builds without Eigen / Ceres / OpenCV).  What
the reference answered is stored in tests/golden/matcher_reference_matrices.npz; the seeded inputs come from
tools/make_golden_matcher.py, which wrote the answers, and are checked against the digests stored beside them.  Bit-exact
match sets on tie-heavy random inputs, with skips, all numBest values, absolute and ratio thresholds, and through the
Hamming distance."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "matcher_reference_matrices.npz")
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_golden_matcher as G  # noqa: E402


@pytest.fixture(scope="module")
def ref():
    return np.load(FIX)


def oracle_set(o):
    return sorted((int(a), int(b), float(d)) for (a, b), d in zip(o["matches"], o["distances"]))


def ref_set(m):
    return [(int(a), int(b), float(d)) for a, b, d in m]


def test_reference_known_answers_on_the_reference_itself(ref, oracle):
    """testMatcher.cpp:69-155 on the compiled reference: the fixture the oracle is pinned with really is what the
    reference computes, and the oracle computes it too."""
    for j, ((D, skipA, use_ratio), want) in enumerate(zip(G.known_answer_inputs(), ({(1, 2), (2, 1), (3, 3)}, {(1, 3), (3, 1)}))):
        got = ref_set(ref["known%d_matches" % j])
        assert {(a, b) for a, b, _ in got} == want
        assert oracle_set(oracle.match_matrix(D, skipA, None, 4.0, 4, use_ratio, 3.0)) == got


@pytest.mark.parametrize("num_best", [1, 2, 4, 8])
@pytest.mark.parametrize("use_ratio", [False, True])
def test_oracle_equals_reference_on_tie_heavy_matrices(ref, oracle, num_best, use_ratio):
    k = "tie%d_%d_" % (num_best, use_ratio)
    trials = G.tie_heavy_trials(num_best, use_ratio)
    assert G.digest(*[a for t in trials for a in t[:3]], np.array([t[3:] for t in trials])) == str(ref[k + "inputs_sha256"]), \
        "inputs differ from those the reference answered on"
    counts, returned, m_all = ref[k + "counts"], ref[k + "returned"], ref[k + "matches"]
    assert len(counts) == len(trials) == 60
    off = 0
    for trial, ((D, skipA, skipB, thr, ratio), cnt, n) in enumerate(zip(trials, counts, returned)):
        r = ref_set(m_all[off:off + cnt])
        off += cnt
        o = oracle.match_matrix(D, skipA, skipB, thr, num_best, use_ratio, ratio)
        assert oracle_set(o) == r, (trial, D.shape, thr)
        assert n == len(r)
    assert off == len(m_all)


def test_oracle_hamming_equals_reference_on_descriptor_distances(ref, oracle):
    lists = G.hamming_lists()
    assert G.digest(*[a for l in lists for a in l]) == str(ref["ham_inputs_sha256"]), "inputs differ from those the reference answered on"
    for j, (A, B) in enumerate(lists):
        for use_ratio in (False, True):
            r = ref_set(ref["ham%d_matches%d" % (j, use_ratio)])
            o = oracle.match_hamming(A, B, None, None, threshold=60.0, num_best=4, use_ratio=use_ratio, ratio_threshold=3.0)
            assert oracle_set(o) == r


def test_four_reference_threads_agree_with_the_sequential_order_on_these_inputs(ref, oracle):
    """The reference runs four matcher threads (Frontend.cpp:80) and its result can depend on their interleaving; the
    project's contract is the sequential order.  On inputs without contested ties the two coincide -- a sanity check that the
    threaded reference is the same algorithm, not a parity requirement."""
    D = G.threads_matrix()
    assert G.digest(D) == str(ref["threads_inputs_sha256"]), "inputs differ from those the reference answered on"
    r1, r4 = ref_set(ref["threads_matches1"]), ref_set(ref["threads_matches4"])
    assert r1 == r4
    assert oracle_set(oracle.match_matrix(D, threshold=30.0)) == r4
