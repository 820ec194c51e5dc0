#!/usr/bin/env python
"""Golden vectors for the matcher produced by the REFERENCE ITSELF: okvis_matcher compiled unmodified from /root/reference
(oracle/Makefile.ref -> oracle/_ref/libokvis_matcher_ref.so, one matcher thread = the sequential order of the project's
contract).  Writes tests/golden/matcher_reference.npz: descriptor lists, skip flags, parameters and the (A, B, distance)
matches DenseMatcher::match emitted.  The reference tree does not exist on the GPU box; the vectors travel instead.
Also writes tests/golden/matcher_reference_matrices.npz: what the reference matcher answers on the seeded inputs of
tests/test_oracle_vs_reference_matcher.py (the fixture of its own testMatcher.cpp, tie-heavy distance matrices, Hamming
distances, four matcher threads) with digests of those inputs, so that the oracle is checked against the reference
without it.
Usage: python tools/make_golden_matcher.py [--check]"""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "matcher_reference.npz")
OUT_MATRICES = os.path.join(ROOT, "tests", "golden", "matcher_reference_matrices.npz")
SO = os.path.join(ROOT, "oracle", "_ref", "libokvis_matcher_ref.so")

CASES = [  # nA, nB, bytes, max flipped bits, skip fraction, threshold, numBest, ratio test, ratio threshold
    (300, 280, 48, 30, 0.05, 60.0, 4, False, 3.0),
    (300, 280, 48, 30, 0.05, 60.0, 4, True, 3.0),
    (64, 400, 48, 60, 0.10, 60.0, 4, False, 3.0),
    (400, 37, 48, 12, 0.00, 60.0, 4, True, 1.5),
    (129, 128, 64, 64, 0.05, 80.0, 4, False, 3.0),
    (200, 200, 48, 8, 0.02, 60.0, 1, False, 3.0),
    (200, 200, 48, 8, 0.02, 60.0, 2, True, 3.0),
    (150, 170, 48, 20, 0.00, 60.0, 8, False, 3.0),
    (1, 1, 48, 0, 0.00, 60.0, 4, False, 3.0),
    (50, 60, 48, 400, 0.00, 60.0, 4, False, 3.0),       # almost nothing below the threshold
]


def make_case(i, spec):
    nA, nB, nbytes, flips, skipf, thr, nb, use_ratio, ratio = spec
    rng = np.random.Generator(np.random.PCG64(0x0B200 + 7000 + i))
    base = rng.integers(0, 256, (max(nA, nB), nbytes), dtype=np.uint8)
    A = base[:nA].copy()
    B = base[rng.permutation(max(nA, nB))[:nB]].copy()
    for row in B:      # few bit flips => many small, tied distances
        for j in rng.integers(0, nbytes * 8, rng.integers(0, flips + 1)):
            row[j >> 3] ^= np.uint8(1 << (j & 7))
    skipA = (rng.random(nA) < skipf).astype(np.uint8)
    skipB = (rng.random(nB) < skipf).astype(np.uint8)
    return A, B, skipA, skipB


def reference_matches(lib, A, B, skipA, skipB, thr, nb, use_ratio, ratio):
    D = np.ascontiguousarray(np.unpackbits(A[:, None, :] ^ B[None, :, :], axis=2).sum(2), np.float32)
    oa, od = np.zeros(len(B), np.int32), np.zeros(len(B), np.float32)
    lib.okr_match(C.c_void_p(D.ctypes.data), len(A), len(B), C.c_void_p(skipA.ctypes.data), C.c_void_p(skipB.ctypes.data), C.c_float(thr), nb,
                  int(use_ratio), C.c_float(ratio), 1, C.c_void_p(oa.ctypes.data), C.c_void_p(od.ctypes.data))
    m = np.array([(int(oa[b]), b, float(od[b])) for b in range(len(B)) if oa[b] >= 0], np.float64).reshape(-1, 3)
    return m


def reference_match_matrix(lib, D, skipA=None, skipB=None, threshold=4.0, num_best=4, use_ratio=False, ratio_threshold=3.0,
                           threads=1):
    """DenseMatcher::match over a distance matrix: the matches sorted as (a, b, distance) rows and the count it returned."""
    D = np.ascontiguousarray(D, np.float32)
    nA, nB = D.shape
    a, d = np.zeros(nB, np.int32), np.zeros(nB, np.float32)
    sa = np.ascontiguousarray(skipA, np.uint8) if skipA is not None else None
    sb = np.ascontiguousarray(skipB, np.uint8) if skipB is not None else None
    n = lib.okr_match(C.c_void_p(D.ctypes.data), nA, nB, C.c_void_p(sa.ctypes.data) if sa is not None else None,
                      C.c_void_p(sb.ctypes.data) if sb is not None else None, C.c_float(threshold), num_best, int(use_ratio),
                      C.c_float(ratio_threshold), threads, C.c_void_p(a.ctypes.data), C.c_void_p(d.ctypes.data))
    m = sorted((int(a[b]), b, float(d[b])) for b in range(nB) if a[b] >= 0)
    return np.array(m, np.float64).reshape(-1, 3), n


def known_answer_inputs():
    """testMatcher.cpp:69-155: (D, skipA, use_ratio) for the absolute threshold, then the ratio test (threshold 4, ratio 3)."""
    def dist(va, vb):
        return np.abs(np.subtract.outer(np.array(va, float), np.array(vb, float))).astype(np.float32)
    return [(dist([1, 3, 2, 0.9], [18, 2.1, 4, 1]), np.array([1, 0, 0, 0], np.uint8), False),
            (dist([8, 1, 3, 2, 0.9], [18, 2.1, 4, 1, 7]), np.array([1, 0, 0, 0, 0], np.uint8), True)]


def tie_heavy_trials(num_best, use_ratio):
    """60 seeded (D, skipA, skipB, threshold, ratio_threshold): few distinct distances, so ties everywhere."""
    rng = np.random.default_rng(100 + num_best + 10 * use_ratio)
    trials = []
    for _ in range(60):
        nA, nB = int(rng.integers(1, 60)), int(rng.integers(1, 60))
        levels = int(rng.integers(2, 12))
        D = rng.integers(0, levels, (nA, nB)).astype(np.float32)
        skipA = (rng.random(nA) < 0.1).astype(np.uint8)
        skipB = (rng.random(nB) < 0.1).astype(np.uint8)
        thr = float(rng.integers(1, levels + 1))
        ratio = float(rng.choice([1.0, 1.5, 3.0]))
        trials.append((D, skipA, skipB, thr, ratio))
    return trials


def hamming_lists():
    """Three seeded pairs of 48-byte descriptor lists, B a permuted copy of A with a few bits flipped per row."""
    rng = np.random.default_rng(7)
    lists = []
    for nA, nB, flips in ((300, 280, 30), (64, 512, 60), (500, 37, 12)):
        base = rng.integers(0, 256, (max(nA, nB), 48), dtype=np.uint8)
        A = base[:nA].copy()
        B = base[rng.permutation(max(nA, nB))[:nB]].copy()
        for row in B:
            for i in rng.integers(0, 384, rng.integers(0, flips)):
                row[i >> 3] ^= np.uint8(1 << (i & 7))
        lists.append((A, B))
    return lists


def hamming_matrix(A, B):
    return np.unpackbits(A[:, None, :] ^ B[None, :, :], axis=2).sum(2).astype(np.float32)


def threads_matrix():
    """Continuous distances, no ties: the one- and four-thread reference agree on it."""
    return np.random.default_rng(11).random((200, 180)).astype(np.float32) * 100.0


def digest(*arrays):
    """SHA-256 over shapes, dtypes and bytes: the stored answers hold only for the inputs they were computed on."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(repr((a.shape, a.dtype.str)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def generate_matrices(lib):
    """The reference's answers on the inputs of tests/test_oracle_vs_reference_matcher.py.  The inputs themselves come
    from the seeded builders above (stored, they would be ~400 kB of incompressible data); each group carries the digest
    of its inputs so that a change of the builders or of NumPy's random streams shows up as such."""
    out = {"source": np.array("okvis_matcher (unmodified reference sources) via oracle/Makefile.ref")}
    for j, (D, sA, use_ratio) in enumerate(known_answer_inputs()):
        out["known%d_matches" % j] = reference_match_matrix(lib, D, skipA=sA, threshold=4.0, use_ratio=use_ratio, ratio_threshold=3.0)[0]
    for num_best in (1, 2, 4, 8):
        for use_ratio in (False, True):
            trials = tie_heavy_trials(num_best, use_ratio)
            res = [reference_match_matrix(lib, D, sA, sB, thr, num_best, use_ratio, ratio) for D, sA, sB, thr, ratio in trials]
            k = "tie%d_%d_" % (num_best, use_ratio)
            out[k + "matches"] = np.concatenate([m for m, _ in res])
            out[k + "counts"] = np.array([len(m) for m, _ in res], np.int32)
            out[k + "returned"] = np.array([n for _, n in res], np.int32)
            out[k + "inputs_sha256"] = np.array(digest(*[a for t in trials for a in t[:3]], np.array([t[3:] for t in trials])))
    lists = hamming_lists()
    for j, (A, B) in enumerate(lists):
        for use_ratio in (False, True):
            out["ham%d_matches%d" % (j, use_ratio)] = reference_match_matrix(lib, hamming_matrix(A, B), None, None, 60.0, 4, use_ratio, 3.0)[0]
    out["ham_inputs_sha256"] = np.array(digest(*[a for l in lists for a in l]))
    D = threads_matrix()
    for t in (1, 4):
        out["threads_matches%d" % t] = reference_match_matrix(lib, D, threshold=30.0, threads=t)[0]
    out["threads_inputs_sha256"] = np.array(digest(D))
    return out


def generate():
    subprocess.run(["make", "-s", "-f", "Makefile.ref"], cwd=os.path.join(ROOT, "oracle"), check=True)
    lib = C.CDLL(SO)
    lib.okr_match.restype = C.c_int
    out = {"n_cases": np.array(len(CASES)), "source": np.array("okvis_matcher (unmodified reference sources, 1 matcher thread) via oracle/Makefile.ref")}
    for i, spec in enumerate(CASES):
        A, B, sA, sB = make_case(i, spec)
        out["A%d" % i], out["B%d" % i], out["skipA%d" % i], out["skipB%d" % i] = A, B, sA, sB
        out["params%d" % i] = np.array([spec[5], spec[6], float(spec[7]), spec[8]])
        out["matches%d" % i] = reference_matches(lib, A, B, sA, sB, spec[5], spec[6], spec[7], spec[8])
    return {OUT: out, OUT_MATRICES: generate_matrices(lib)}


def main():
    outs = generate()
    if "--check" in sys.argv:
        for path, out in outs.items():
            old = np.load(path)
            for k in out:
                if k != "source":
                    assert np.array_equal(out[k], old[k]), (path, k)
        print("fixtures reproduced")
        return
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    for path, out in outs.items():
        np.savez_compressed(path, **out)
        print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
