"""Generate tests/golden/native_vectors.npz and reference_trials.npz from the REFERENCE's own compiled natives
(oracle/_ref, built by oracle/build_ref.py from /root/reference).  Run in the build container:

    python oracle/build_ref.py && python tests/golden/make_golden.py

The vectors pin the oracle (tests/test_oracle.py) and, on the GPU box where /root/reference does not
exist, the CUDA kernels (tests/test_gpu_golden.py)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import build_ref  # noqa: E402

TRIAL_MSS_PARAMS = ((0, -1), (3, 2), (50, 50))


def reference_trials():
    """The seeded inputs of tests/test_oracle.py::test_oracle_against_compiled_reference: 40 trials of
    (scores, labels, text)."""
    rng = np.random.default_rng(9)
    for _ in range(40):
        n = int(rng.integers(1, 3000))
        s = rng.normal(size=n) * 3 - rng.random()
        lab = rng.integers(0, 5, size=n)
        text = "".join(np.array(list("ACGTNacgtnX"))[rng.integers(0, 11, size=n)])
        yield s, lab, text


def trial_vectors(seq, mss):
    """find_mss_labels (as its argmax: the rows are one-hot), one_hot_encode_dna_sequence and yield_segments of
    `seq` / `mss` (the reference modules, or the oracle) on reference_trials()."""
    out = {}
    for i, (s, lab, text) in enumerate(reference_trials()):
        for k, (ml, xd) in enumerate(TRIAL_MSS_PARAMS):
            res = np.asarray(mss.find_mss_labels(s, lab, 5, ml, xd))
            assert ((res == 0) | (res == 1)).all() and (res.sum(axis=1) == 1).all()
            out["mss_%d_%d" % (i, k)] = res.argmax(axis=1).astype(np.uint8)
        if set(text) != {"N"}:
            st, fwd = seq.one_hot_encode_dna_sequence(text)
            out["enc_start_%d" % i] = np.int64(st)
            out["enc_fwd_%d" % i] = np.asarray(fwd)
        out["seg_%d" % i] = np.array(list(seq.yield_segments(lab, 5)), dtype=np.int64).reshape(-1, 3)
    out["n"] = np.int64(i + 1)
    return out


def main():
    assert build_ref.build(), "reference natives unavailable"
    ref_seq, ref_mss = build_ref.load()
    rng = np.random.default_rng(20240611)
    out = {}
    # ---- one_hot_encode_dna_sequence (deepgrp/sequence.pyx:55-58)
    texts = ["ACGT", "acgtnACGTN", "NNNACGTNNN", "nnACGTnn", "NNNNACGTRYKMNNN", "A", "", "NACGTXN",
             "N" * 17 + "".join(np.array(list("ACGTNacgtnRYKM-*"))[rng.integers(0, 16, size=997)]) + "NN"]
    for i, t in enumerate(texts):
        st, fwd = ref_seq.one_hot_encode_dna_sequence(t)
        out["enc_text_%d" % i] = np.frombuffer(t.encode(), dtype=np.uint8)
        out["enc_start_%d" % i] = np.int64(st)
        out["enc_fwd_%d" % i] = fwd
    out["enc_n"] = np.int64(len(texts))
    # ---- get_max (deepgrp/sequence.pyx:67-76 -> maxcalc.c)
    cases = [(7, 30, 5, 10), (3, 10, 5, 10), (5, 13, 4, 1), (4, 20, 5, 37)]
    for i, (b, t, c, s) in enumerate(cases):
        inputs = rng.random((b, t, c), dtype=np.float32)
        base = (rng.random(((b - 1) * s + t + 5, c), dtype=np.float32) * 0.5).astype(np.float32)
        res = ref_seq.get_max(base.copy(), inputs, s)
        out["max_in_%d" % i] = inputs
        out["max_base_%d" % i] = base
        out["max_stride_%d" % i] = np.int64(s)
        out["max_out_%d" % i] = res
    out["max_n"] = np.int64(len(cases))
    # ---- yield_segments / get_segments (deepgrp/sequence.pyx:40-53, 79-85)
    labs = [np.array([0], np.int64), np.array([3], np.int64), np.array([2, 2], np.int64),
            np.array([0, 0, 2], np.int64), np.array([2, 2, 0], np.int64),
            np.repeat(rng.integers(0, 5, size=300), rng.integers(1, 9, size=300)).astype(np.int64),
            np.zeros(50, np.int64), np.full(50, 4, np.int64)]
    for i, lab in enumerate(labs):
        segs = np.array(list(ref_seq.yield_segments(lab, 11)), dtype=np.int64).reshape(-1, 3)
        out["seg_lab_%d" % i] = lab
        out["seg_out_%d" % i] = segs
    out["seg_n"] = np.int64(len(labs))
    # ---- find_mss_labels (deepgrp/_mss/pymss.pyx:16-27 -> mss.c)
    k = 0
    for n in (1, 14, 200, 5000):
        for kind in range(5):
            if kind == 0:
                s = rng.normal(size=n)
            elif kind == 1:
                s = rng.normal(size=n) - 0.5
            elif kind == 2:
                s = rng.integers(-3, 4, size=n).astype(np.float64)
            elif kind == 3:
                s = np.where(rng.random(n) < 0.05, 13.2, -1.32) * (1 + 1e-3 * rng.normal(size=n))
            else:
                lab_runs = np.repeat(rng.integers(0, 5, size=n), rng.integers(1, 60, size=n))[:n]
                s = np.where(lab_runs > 0, 4.59, -45.9) * rng.random(n)
            lab = np.repeat(rng.integers(0, 5, size=n), rng.integers(1, 7, size=n))[:n].astype(np.int64)
            for (ml, xd) in ((0, -1), (1, 0), (2, 3), (50, 50)):
                res = ref_mss.find_mss_labels(np.ascontiguousarray(s, dtype=np.float64), lab, 5, ml, xd)
                out["mss_s_%d" % k] = np.asarray(s, dtype=np.float64)
                out["mss_lab_%d" % k] = lab
                out["mss_par_%d" % k] = np.array([ml, xd], np.int64)
                out["mss_out_%d" % k] = np.asarray(res).argmax(axis=1).astype(np.uint8)
                assert (np.asarray(res).sum(axis=1) == 1).all()
                k += 1
    out["mss_n"] = np.int64(k)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_trials.npz")
    np.savez_compressed(path, **trial_vectors(ref_seq, ref_mss))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
