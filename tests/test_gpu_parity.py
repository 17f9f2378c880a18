"""GPU parity tests: the CUDA path (through the C ABI / the Python mirror of the reference API)
against the CPU oracle on the same seeded inputs.  Integer/byte/index work is bit-exact; the
floating-point forward is within 1e-3 absolute on probabilities (BASELINE.json north_star) -- the
tests assert the much tighter 2e-5 -- and >= 99.99 % identical labels."""
import ctypes
import io

import numpy as np
import pytest

from conftest import messy_fasta, random_dna, write_fasta

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-3        # north_star tolerance
PROB_TOL_TIGHT = 2e-5  # what fp32 FFMA arithmetic should achieve


@pytest.fixture(scope="module")
def dg(gpu_ctx):
    import deepgrp_b200.sequence as seq
    import deepgrp_b200.mss as mss
    import deepgrp_b200.prediction as pred
    import deepgrp_b200.model as model

    class NS:
        pass
    ns = NS()
    ns.seq, ns.mss, ns.pred, ns.model, ns.ctx = seq, mss, pred, model, gpu_ctx
    return ns


# ------------------------------------------------------------------ encode
@pytest.mark.parametrize("text", [
    "ACGT", "acgtnACGTN", "NNNACGTNNN", "nnACGTnn", "NNNNACGTRYKMNNN", "A", "", "NACGTXN",
    "ACGT" * 1000 + "N" * 77, "N" * 50 + "acgtryswkm" * 333 + "N",
])
def test_one_hot_matches_oracle(dg, oracle, text):
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    st_o, fwd_o = oracle.one_hot_encode_dna_sequence(text)
    assert st == st_o
    assert fwd.dtype == np.int8 and fwd.shape == fwd_o.shape
    assert np.array_equal(fwd, fwd_o)


def test_one_hot_reference_known_answer(dg):
    # reference tests/test_sequence.py:10-28
    rng = np.random.default_rng(3)
    letters = np.array(list("ACGTN"))
    seq = "".join(letters[rng.integers(0, 5, size=5000)])
    seq = "NNNN" + "A" + seq + "C" + "NNN"
    st, fwd = dg.seq.one_hot_encode_dna_sequence(seq)
    assert st == 4
    assert fwd.shape == (5, len(seq) - 7)
    assert (fwd.sum(axis=0) == 1).all()
    expected = np.array(["ACGTN".index(c) for c in seq[4:-3]])
    assert np.array_equal(fwd.argmax(axis=0), expected)


def test_one_hot_all_n_raises(dg):
    with pytest.raises(ValueError):
        dg.seq.one_hot_encode_dna_sequence("NNNNNN")


def test_one_hot_large(dg, oracle):
    text = "N" * 1234 + random_dna(3_000_017, 11, "ACGTNacgtnRY") + "N" * 999
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    st_o, fwd_o = oracle.one_hot_encode_dna_sequence(text)
    assert st == st_o and np.array_equal(fwd, fwd_o)


# ------------------------------------------------------------------ get_max
def test_get_max_reference_known_answer(dg):
    # reference tests/test_sequence.py:47-56
    inputs = np.zeros((10, 100, 5), dtype=np.float32)
    for i in range(10):
        inputs[i] = i + 1
    out = np.zeros((1000, 5), dtype=np.float32)
    ret = dg.seq.get_max(out, inputs, 50)
    assert ret is out
    exp = np.zeros((1000, 5), dtype=np.float32)
    for i in range(10):
        exp[i * 50:i * 50 + 100] = np.maximum(exp[i * 50:i * 50 + 100], i + 1)
    assert np.array_equal(out, exp)


@pytest.mark.parametrize("b,t,c,stride", [(7, 150, 5, 50), (3, 10, 5, 10), (5, 33, 4, 1), (4, 20, 5, 37),
                                          (256, 342, 5, 50)])
def test_get_max_matches_oracle(dg, oracle, b, t, c, stride):
    rng = np.random.default_rng(b * 1000 + t)
    inputs = rng.random((b, t, c), dtype=np.float32)
    rows = (b - 1) * stride + t + 13
    base = rng.random((rows, c), dtype=np.float32) * 0.5
    out = base.copy()
    exp = oracle.get_max(base.copy(), inputs, stride)
    dg.seq.get_max(out, inputs, stride)
    assert np.array_equal(out, exp)


def test_get_max_dtype_errors(dg):
    with pytest.raises(ValueError):
        dg.seq.get_max(np.zeros((10, 5)), np.zeros((1, 5, 5), np.float32), 1)
    with pytest.raises(TypeError):
        dg.seq.get_max(None, np.zeros((1, 5, 5), np.float32), 1)


# ------------------------------------------------------------------ segments
def test_segments_reference_cases(dg, oracle):
    # reference tests/test_sequence.py:30-44: one run of `label` at [start, start+len)
    for start in (0, 1, 50, 90):
        for length in (1, 5, 10):
            for label in (1, 2, 4):
                classes = np.zeros(100, dtype=np.int64)
                classes[start:start + length] = label
                got = dg.seq.get_segments(classes, 0)
                assert got == oracle.get_segments(classes, 0)


@pytest.mark.parametrize("n,seed", [(1, 0), (2, 1), (3, 2), (100, 3), (4097, 4), (100_000, 5)])
def test_yield_segments_matches_oracle(dg, oracle, n, seed):
    rng = np.random.default_rng(seed)
    # runs of random labels with random lengths
    lab = np.repeat(rng.integers(0, 5, size=n), rng.integers(1, 9, size=n))[:n].astype(np.int64)
    for arr in (lab, np.zeros(n, np.int64), np.full(n, 3, np.int64)):
        got = list(dg.seq.yield_segments(arr, 17))
        exp = list(oracle.yield_segments(arr, 17))
        assert got == exp
        for s in (0, n // 2, n - 1):
            assert dg.seq.get_segments(arr, s) == oracle.get_segments(arr, s)


# ------------------------------------------------------------------ MSS
def test_mss_reference_known_answer(dg, oracle):
    # reference tests/test_mss.py:10-24 style: 14-element vector, min_mss_len 0/1, xdrop -1/0/10
    scores = np.array([4.0, -5, 3, -3, 1, 2, -2, 2, -2, 1, 5, -5, -1, 3], dtype=np.float64)
    labels = np.array([1, 0, 2, 0, 2, 2, 0, 3, 0, 3, 3, 0, 0, 1], dtype=np.int64)
    for min_len in (0, 1, 2):
        for xdrop in (-1, 0, 10):
            got = dg.mss.find_mss_labels(scores, labels, 5, min_len, xdrop)
            exp = oracle.find_mss_labels(scores, labels, 5, min_len, xdrop)
            assert np.array_equal(got, exp)


def _score_sets(rng, n):
    yield "normal", rng.normal(size=n)
    yield "neg", rng.normal(size=n) - 0.5
    yield "pos", rng.normal(size=n) + 0.3
    yield "ties", rng.integers(-3, 4, size=n).astype(np.float64)
    yield "sparse", np.where(rng.random(n) < 0.05, 13.2, -1.32) * (1 + 1e-3 * rng.normal(size=n))
    yield "f32", (rng.normal(size=n) * 3).astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("n", [1, 2, 17, 1000, 65_537])
@pytest.mark.parametrize("chunk", [0, 32, 64])
def test_mss_find_all_bit_exact(dg, oracle, n, chunk):
    rng = np.random.default_rng(n + chunk)
    dg.ctx.set_int("mss_chunk", chunk)
    try:
        for name, s in _score_sets(rng, n):
            for xdrop in (-1.0, 3.0, 40.0):
                for min_sc in (0.0, 2.7, 25.0):
                    got = dg.mss.mss_find_all(s, min_sc, xdrop)
                    exp = oracle.mss_find_all(s, min_sc, xdrop)
                    assert got.size == exp.size, (name, xdrop, min_sc)
                    assert np.array_equal(got["st"], exp["st"]) and np.array_equal(got["en"], exp["en"])
                    assert np.array_equal(got["sc"].view(np.int64), exp["sc"].view(np.int64))
    finally:
        dg.ctx.set_int("mss_chunk", 0)


def test_find_mss_labels_matches_oracle_large(dg, oracle):
    rng = np.random.default_rng(77)
    n = 300_000
    lab = np.repeat(rng.integers(0, 5, size=n), rng.integers(1, 200, size=n))[:n].astype(np.int64)
    t = np.float32(np.log(0.99 / 0.01))
    scores = np.where(lab > 0, t, -10 * t).astype(np.float64) * rng.random(n)
    for min_len, xdrop in ((50, 50), (0, 50), (50, -1), (5, 2)):
        got = dg.mss.find_mss_labels(scores, lab, 5, min_len, xdrop)
        exp = oracle.find_mss_labels(scores, lab, 5, min_len, xdrop)
        assert np.array_equal(got, exp)


def _long_segment_case(rng, lengths, gap=3):
    """Scores whose maximal segments are exactly the given positive runs (float32-valued; runs separated by `gap`
    positions negative enough that no two runs merge), labels with zeros to fill in every run."""
    t = float(np.float32(np.log(0.99 / 0.01)))
    scores, labels = [], []
    for k, ln in enumerate(lengths):
        scores.append(np.full(ln, t)); scores.append(np.full(gap, -float(2 ** 24)))
        lab = rng.integers(0, 5, size=ln)
        lab[rng.random(ln) < 0.5] = 0
        if k % 3 == 1:
            lab[lab == 1] = 0                   # the majority is not class 1
        if k % 5 == 4:
            lab[:] = 0                          # no positive label at all: default class 1
        labels.append(lab); labels.append(np.zeros(gap, dtype=lab.dtype))
    return np.concatenate(scores), np.concatenate(labels).astype(np.int64)


@pytest.mark.parametrize("lengths", [
    [200_000],                                   # one segment spanning many blocks
    [8192, 8193, 8191, 50, 16_384, 16_385, 3, 70_000, 8193],   # both sides of the long-segment threshold
    [100, 30_000, 60, 60, 60, 9000, 9000, 20, 123_457, 51],
])
def test_gap_fill_long_segments(dg, oracle, lengths):
    """Segments longer than a warp should walk alone (mss.cu: gap_long_kernel): label counts and the fill of
    segments that span many blocks, start and end anywhere, next to short ones -- int64 labels through
    find_mss_labels, uint8 labels + float32 scores through dgrp_finish_record."""
    from deepgrp_b200 import sharding
    rng = np.random.default_rng(len(lengths))
    scores, labels = _long_segment_case(rng, lengths)
    for min_len, xdrop in ((50, 50), (1, -1)):
        exp = oracle.find_mss_labels(scores, labels, 5, min_len, xdrop)
        got = dg.mss.find_mss_labels(scores, labels, 5, min_len, xdrop)
        assert np.array_equal(got, exp)
        out, rows = sharding.finish_record(labels.astype(np.uint8), scores.astype(np.float32), 5, True, min_len,
                                           xdrop, 7)
        assert np.array_equal(out, exp.argmax(axis=1).astype(np.uint8))
        exp_rows = [(a, b, l) for a, b, l in oracle.yield_segments(exp.argmax(axis=1).astype(np.int64), 7) if l > 0]
        assert list(zip(rows["start"].tolist(), rows["end"].tolist(), rows["label"].tolist())) == exp_rows


# ------------------------------------------------------------------ score transform / softmax
def test_mss_scores_and_softmax(dg, oracle):
    rng = np.random.default_rng(5)
    probs = rng.dirichlet(np.ones(5) * 0.3, size=20_000).astype(np.float32)
    probs[:100] = 0.0                       # never-covered rows
    probs[100:200] = [0.2, 0.2, 0.2, 0.2, 0.2]   # ties -> class 0
    sc, cl = dg.pred.mss_scores(probs)
    sc_o, cl_o = oracle.apply_mss_scores(probs)
    assert np.array_equal(cl, cl_o)
    # device logf vs numpy float32 log may differ by an ulp (SURVEY.md section 8a item 6)
    assert np.allclose(sc, sc_o, rtol=3e-7, atol=1e-6)
    assert abs(sc[0] - 138.155) < 1e-2
    sm = dg.pred.softmax(probs)
    sm_o = oracle.softmax(probs)
    assert np.allclose(sm, sm_o, rtol=1e-6, atol=1e-7)
    assert np.array_equal(sm.argmax(axis=1), sm_o.argmax(axis=1))


def test_apply_mss_matches_oracle_given_scores(dg, oracle):
    """MSS bit-exact given identical score inputs: feed the GPU's own scores to the oracle."""
    rng = np.random.default_rng(6)
    n = 200_000
    lab = np.repeat(rng.integers(0, 5, size=n), rng.integers(1, 300, size=n))[:n]
    conf = rng.random(n).astype(np.float32) * 0.6 + 0.39
    probs = np.full((n, 5), 0.0, np.float32)
    probs[np.arange(n), lab] = conf
    rest = (1 - conf) / 4
    for c in range(5):
        probs[np.arange(n), c] = np.where(lab == c, conf, rest)
    from deepgrp_b200.model import Options
    opt = Options(min_mss_len=50, xdrop_len=50)
    got = dg.pred.apply_mss(probs, opt)
    sc, cl = dg.pred.mss_scores(probs)
    exp = oracle.find_mss_labels(sc, cl, 5, 50, 50)
    assert np.array_equal(got, exp)


# ------------------------------------------------------------------ forward
@pytest.mark.parametrize("T,U,attention", [(150, 32, True), (60, 60, True), (40, 16, False),
                                           (50, 50, True), (30, 100, True), (37, 7, True)])
def test_forward_windows_matches_oracle(dg, oracle, T, U, attention):
    w = dg.model.random_weights(T, U, attention=attention, seed=1)
    rng = np.random.default_rng(T + U)
    codes = rng.integers(0, 5, size=(70, T))
    batch = np.eye(5, dtype=np.float32)[codes]
    got = w.predict_on_batch(batch)
    exp = oracle.model_forward(batch, w.as_dict())
    assert got.shape == exp.shape
    assert np.abs(got - exp).max() < PROB_TOL_TIGHT
    # scaled weights: confident outputs
    w4 = w.scaled(4.0)
    got4 = w4.predict_on_batch(batch)
    exp4 = oracle.model_forward(batch, w4.as_dict())
    assert np.abs(got4 - exp4).max() < PROB_TOL_TIGHT


def test_forward_dense_non_onehot_input(dg, oracle):
    w = dg.model.random_weights(48, 32, attention=True, seed=2)
    rng = np.random.default_rng(0)
    batch = rng.random((9, 48, 5), dtype=np.float32)
    got = w.predict_on_batch(batch)
    exp = oracle.model_forward(batch, w.as_dict())
    assert np.abs(got - exp).max() < PROB_TOL_TIGHT


@pytest.mark.parametrize("L,T,U,step,B", [(5000, 150, 32, 50, 16), (3000, 150, 32, 50, 256),
                                          (2000, 100, 60, 33, 7), (150, 150, 32, 50, 16),
                                          (151, 150, 32, 50, 16), (100, 150, 32, 50, 16)])
def test_predict_matches_oracle_including_partial_batch(dg, oracle, L, T, U, step, B):
    w = dg.model.random_weights(T, U, attention=True, seed=3).scaled(3.0)
    text = random_dna(L, L + step, "ACGTN")
    text = "A" + text[1:-1] + "C"
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    ds = dg.pred.fetch_validation_batch(fwd, step, B, T)
    got = dg.pred.predict(w, ds, (fwd.shape[1], 5), step)
    exp = oracle.predict(lambda b: oracle.model_forward(b, w.as_dict()),
                         oracle.fetch_validation_batch(fwd, step, B, T), (fwd.shape[1], 5), step)
    assert got.shape == exp.shape
    assert np.abs(got - exp).max() < PROB_TOL_TIGHT
    assert np.array_equal(got == 0, exp == 0)            # identical coverage (incl. misplaced tail)
    fixed = dg.pred.predict(w, ds, (fwd.shape[1], 5), step, compat="fixed")
    n_win = len(range(0, fwd.shape[1] - T, step))
    if n_win % B:
        assert not np.array_equal(fixed == 0, exp == 0) or n_win < B


def test_predict_generic_route_equals_fused(dg):
    """The literal reference loop (iterate batches, predict_on_batch, get_max) and the fused call."""
    w = dg.model.random_weights(150, 32, attention=True, seed=4)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(random_dna(4000, 9))
    ds = dg.pred.fetch_validation_batch(fwd, 50, 16, 150)
    fused = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)

    class Wrapped:       # hides the ModelWeights type -> generic route
        def predict_on_batch(self, batch):
            return w.predict_on_batch(batch)
    generic = dg.pred.predict(Wrapped(), iter(ds), (fwd.shape[1], 5), 50)
    # the fused call runs the tcgen05 recurrence, predict_on_batch the fp32 FFMA kernel
    assert np.abs(fused - generic).max() < 2e-5   # random-init weights; half-precision score scratch
    assert np.array_equal(fused == 0, generic == 0)
    dg.ctx.set_int("forward_tc", 0)
    try:
        fused_fp32 = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
    finally:
        dg.ctx.set_int("forward_tc", 1)
    assert np.array_equal(fused_fp32, generic)      # same kernel arithmetic: bit-identical


@pytest.mark.parametrize("T,U", [(150, 32), (342, 60), (64, 16), (100, 50)])
def test_tensor_core_forward_is_fp32_faithful(dg, oracle, T, U):
    """tcgen05 forward (two scaled fp16 pieces per operand, three products) against the float64 oracle on
    x4-scaled weights (sharp attention, all classes present).  The half-precision h_fwd + h_rc scratch
    only perturbs the attention scores: <= 1e-4 on a probability (north_star's bar is 1e-3), labels
    identical to 1e-4."""
    w = dg.model.random_weights(T, U, attention=True, seed=7).scaled(4.0)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(random_dna(12_000, T + U))
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    tc = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
    assert dg.ctx.get_int("forward_used_tc") == 1
    ref64 = oracle.predict(lambda b: oracle.model_forward(b, w.as_dict(), dtype=np.float64).astype(np.float32),
                           oracle.fetch_validation_batch(fwd, 50, 256, T), (fwd.shape[1], 5), 50)
    assert np.abs(tc - ref64).max() < 1e-4
    assert (tc.argmax(axis=1) != ref64.argmax(axis=1)).mean() <= 1e-4


@pytest.mark.parametrize("T,U,step,L", [(512, 40, 50, 9_000),     # scores of 64 windows do not fit: passes of 32
                                        (151, 32, 50, 6_000),     # odd window: one priming round
                                        (342, 60, 7, 3_000),      # small step: dense overlap in the gather
                                        (150, 32, 200, 30_000),   # step > T: uncovered gaps between windows
                                        (33, 20, 50, 4_000),      # window barely longer than a warp
                                        (342, 60, 250, 40_000)])  # largest staged span per tile
def test_tensor_core_forward_shapes(dg, oracle, T, U, step, L):
    """Shapes that exercise the kernel's less travelled paths, against the float64 oracle."""
    w = dg.model.random_weights(T, U, attention=True, seed=11).scaled(2.0)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(random_dna(L, T + step))
    ds = dg.pred.fetch_validation_batch(fwd, step, 16, T)
    tc = dg.pred.predict(w, ds, (fwd.shape[1], 5), step)
    assert dg.ctx.get_int("forward_used_tc") == 1
    ref64 = oracle.predict(lambda b: oracle.model_forward(b, w.as_dict(), dtype=np.float64).astype(np.float32),
                           oracle.fetch_validation_batch(fwd, step, 16, T), (fwd.shape[1], 5), step)
    assert np.array_equal(tc == 0, ref64 == 0)          # the same rows are covered
    assert np.abs(tc - ref64).max() < 2e-5
    assert (tc.argmax(axis=1) != ref64.argmax(axis=1)).mean() <= 1e-4


@pytest.mark.parametrize("compat", ["reference", "fixed"])
def test_vote_gather_equals_atomic_vote(dg, compat):
    """The two forms of the max-vote (window probabilities + gather pass, and atomicMax from inside the
    forward kernel) are the same exact maximum: bit-identical predictions, including the displaced
    last batch of the reference placement and a range call that does not start at row 0."""
    from deepgrp_b200 import sharding
    T, U, L = 150, 32, 23_457
    w = dg.model.random_weights(T, U, attention=True, seed=21).scaled(3.0)
    codes = np.random.default_rng(8).integers(0, 4, size=L, dtype=np.uint8)
    out = {}
    for g in (1, 0):
        dg.ctx.set_int("forward_gather", g)
        try:
            whole = sharding.predict_range(w, codes, L, 0, L, 50, 48, compat={"reference": 0, "fixed": 1}[compat])
            part = sharding.predict_range(w, codes, L, 7_001, 19_990, 50, 48, compat={"reference": 0, "fixed": 1}[compat])
        finally:
            dg.ctx.set_int("forward_gather", 1)
        out[g] = (whole, part)
    for a, b in zip(out[1], out[0]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(out[1][0][0][7_001:19_990], out[1][1][0])
    assert np.array_equal(out[1][0][1][7_001:19_990], out[1][1][1])


def test_tensor_core_forward_random_init_regime(dg, oracle):
    """The benchmark's regime (random-init weights, near-uniform outputs, class margins ~1e-4): the
    default forward must be float32-faithful there, or labels flip."""
    T, U = 342, 60
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(random_dna(20_000, 77))
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    tc = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
    assert dg.ctx.get_int("forward_used_tc") == 1
    ref64 = oracle.predict(lambda b: oracle.model_forward(b, w.as_dict(), dtype=np.float64).astype(np.float32),
                           oracle.fetch_validation_batch(fwd, 50, 256, T), (fwd.shape[1], 5), 50)
    assert np.abs(tc - ref64).max() < 1e-6
    assert (tc.argmax(axis=1) != ref64.argmax(axis=1)).mean() <= 1e-4


# ------------------------------------------------------------------ end to end
def _labels_agree(a, b):
    return float((a == b).mean())


def test_predict_sequence_vs_oracle_labels_and_rows(dg, oracle):
    T, U = 150, 32
    for scale in (1.0, 4.0):
        w = dg.model.random_weights(T, U, attention=True, seed=0).scaled(scale)
        text = "NNNNN" + random_dna(60_000, 21, "ACGTacgtN") + "NN"
        labels, startpos, rows = dg.pred.predict_sequence(w, text.encode(), 50, 256, True, 50, 50)
        lab_o, st_o, probs_o = oracle.predict_record(text.upper(), w.as_dict(), T, 256, 50, True,
                                                     return_probs=True)
        assert startpos == st_o == 5
        assert labels.shape == lab_o.shape
        assert _labels_agree(labels, lab_o) >= 0.9999
        # rows == yield_segments of OUR labels, label > 0 (bit-exact given identical labels)
        exp_rows = [(s, e, l) for s, e, l in oracle.yield_segments(labels.astype(np.int64), startpos) if l > 0]
        got_rows = list(zip(rows["start"].tolist(), rows["end"].tolist(), rows["label"].tolist()))
        assert got_rows == exp_rows
        # no-MSS branch
        labels2, _, _ = dg.pred.predict_sequence(w, text.encode(), 50, 256, False, 50, 50)
        lab2_o, _ = oracle.predict_record(text.upper(), w.as_dict(), T, 256, 50, False)
        assert _labels_agree(labels2, lab2_o) >= 0.9999


def test_stepwise_cli_route_equals_fused(dg, tmp_path):
    from deepgrp_b200.__main__ import _predict, _read_multi_fasta
    from deepgrp_b200.model import Options
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    text = "NN" + random_dna(20_000, 5, "ACGTN") + "N"
    opt = Options(min_mss_len=50, batch_size=256, xdrop_len=50, vecsize=150)
    lab_a, st_a = _predict(text, w, opt, 50, True)
    lab_b, st_b, _ = dg.pred.predict_sequence(w, text.encode(), 50, 256, True, 50, 50)
    assert st_a == st_b
    assert np.array_equal(lab_a, lab_b)


def test_predict_fasta_tsv_vs_oracle(dg, oracle, tmp_path):
    T, U = 150, 32
    w = dg.model.random_weights(T, U, attention=True, seed=0).scaled(4.0)
    recs = [("chrA description text", "NNN" + random_dna(30_000, 1, "ACGTacgtn") + "NNNN"),
            ("chrB", random_dna(140, 2)),                       # shorter than one window
            ("chrC", random_dna(12_345, 3, "ACGTRYKM"))]
    path = tmp_path / "in.fa"
    write_fasta(str(path), recs, width=60)
    raw = open(path, "rb").read()
    got = dg.pred.predict_fasta_tsv(w, raw, str(path), 50, 256, True, 50, 50)
    exp = oracle.predict_fasta_tsv(str(path), w.as_dict(), T)
    got_rows, exp_rows = got.splitlines(), exp.splitlines()
    # identical up to label flips at the 1e-4 level: compare covered bases per (record, label)
    def cover(rows):
        d = {}
        for r in rows:
            f, h, s, e, l = r.split("\t")
            d[(h, l)] = d.get((h, l), 0) + int(e) - int(s)
        return d
    cg, ce = cover(got_rows), cover(exp_rows)
    assert set(cg) == set(ce)
    total = sum(ce.values())
    diff = sum(abs(cg[k] - ce[k]) for k in ce)
    assert diff <= max(2, 2e-4 * total)
    # the GPU-formatted text equals Python formatting of the rows, byte for byte
    rows, records = dg.pred.predict_fasta(w, raw, 50, 256, True, 50, 50)
    assert [r[0] for r in records] == [h for h, _ in recs]
    assert [r[1] for r in records] == [3, 0, 0]
    text = "".join("%s\t%s\t%d\t%d\t%d\n" % (str(path), records[r][0], s, e, l) for s, e, l, r in
                   zip(rows["start"].tolist(), rows["end"].tolist(), rows["label"].tolist(),
                       rows["record"].tolist()))
    assert text == got
    # CRLF line ends, a record with empty header (dropped) and text before the first '>' (dropped)
    raw2 = b"ACGTACGT\r\n>\r\nACGT\r\n" + raw.replace(b"\n", b"\r\n")
    got2 = dg.pred.predict_fasta_tsv(w, raw2, str(path), 50, 256, True, 50, 50)
    assert got2 == got
    with pytest.raises(IndexError):
        dg.pred.predict_fasta_tsv(w, b">x\nACGT\n\nACGT\n", "f", 50, 256, True, 50, 50)
    with pytest.raises(ValueError):
        dg.pred.predict_fasta_tsv(w, b">x\nNNNN\n", "f", 50, 256, True, 50, 50)


@pytest.mark.parametrize("seed", range(24))
def test_fasta_decode_messy_text_equals_python_reader(dg, seed):
    """The GPU FASTA decode against `_read_multi_fasta` (reference deepgrp/__main__.py:20-43) on hostile text:
    same records (header, trimmed length, startpos), and the rows of the messy file equal those of the same
    records written canonically -- identical decoded bytes give bit-identical rows."""
    from deepgrp_b200.__main__ import _read_multi_fasta
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    text = messy_fasta(seed)
    try:
        exp = list(_read_multi_fasta(io.StringIO(text, newline=None)))
    except IndexError:
        with pytest.raises(IndexError):
            dg.pred.predict_fasta(w, text.encode(), 50, 256, True, 50, 50)
        return
    rows, records = dg.pred.predict_fasta(w, text.encode(), 50, 256, True, 50, 50)
    assert [r[0] for r in records] == [h for h, _ in exp]
    for (_, startpos, length), (_, seq) in zip(records, exp):
        assert startpos == len(seq) - len(seq.lstrip("N"))
        assert length == len(seq.strip("N"))
    # whitespace kept inside a line encodes like any non-ACGT byte (channel 4): 'X' stands in for it so that
    # the canonical line breaks cannot strip it
    canon = "".join(">%s\n%s\n" % (h, "\n".join(q[i:i + 60] for i in range(0, len(q), 60)))
                    for h, q in ((h, "".join("X" if c.isspace() else c for c in q)) for h, q in exp))
    rows_c, records_c = dg.pred.predict_fasta(w, canon.encode(), 50, 256, True, 50, 50)
    assert [r[1:] for r in records_c] == [r[1:] for r in records]
    assert np.array_equal(rows, rows_c)


@pytest.mark.parametrize("lead,trail,offset", [(0, 0, 0), (3, 5, 1), (17, 33, 7), (4096, 1, 15), (100_003, 70_001, 3)])
def test_one_hot_trim_unaligned_and_long_n_runs(dg, lead, trail, offset):
    """Edge-N trim with 16-byte loads: N runs longer than a vector / a block, records that start at an odd
    address inside a multi-FASTA buffer (`offset` bases of a first record in front)."""
    body = random_dna(5000, lead + trail, "ACGTN")
    body = "A" + body + "C"
    seq = "N" * lead + body + "N" * trail
    st, fwd = dg.seq.one_hot_encode_dna_sequence(seq)
    assert st == lead and fwd.shape == (5, len(body))
    w = dg.model.random_weights(150, 32, attention=True, seed=0)
    text = ">a\n" + "ACGTACGTACGTACGTA"[:offset + 1] + "\n>b\n" + seq + "\n"
    _, records = dg.pred.predict_fasta(w, text.encode(), 50, 256, False, 50, 50)
    assert records[1] == ("b", lead, len(body))


def test_predict_range_shards_equal_whole(dg):
    """Multi-GPU sharding unit: label/score of disjoint position ranges computed independently
    (with halo re-computation) equal the whole-record result, including the misplaced tail batch."""
    from deepgrp_b200 import _lib
    T, U = 150, 32
    w = dg.model.random_weights(T, U, attention=True, seed=0).scaled(4.0)
    text = random_dna(40_000, 8)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    codes = fwd.argmax(axis=0).astype(np.uint8)
    L = codes.size
    h = w.device_handle(dg.ctx)

    def run(p0, p1, lo, hi):
        lab = np.zeros(p1 - p0, np.uint8)
        sc = np.zeros(p1 - p0, np.float32)
        sub = np.ascontiguousarray(codes[lo:hi])
        _lib.check(_lib.lib().dgrp_predict_range(dg.ctx.handle, h, _lib.ptr(sub), lo, hi - lo, L, p0, p1,
                                                  50, 256, 0, _lib.ptr(lab), _lib.ptr(sc)))
        return lab, sc
    whole_l, whole_s = run(0, L, 0, L)
    cuts = [0, 9_973, 20_000, 33_333, L]
    parts = [run(a, b, 0, L) for a, b in zip(cuts[:-1], cuts[1:])]
    assert np.array_equal(np.concatenate([p[0] for p in parts]), whole_l)
    assert np.array_equal(np.concatenate([p[1] for p in parts]).view(np.int32), whole_s.view(np.int32))


def test_contig_sharding_equals_single_rank(dg, tmp_path):
    """Every rank decodes the file and computes only its records; merged texts == single-rank text."""
    from deepgrp_b200 import sharding
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    recs = [("r%d" % i, random_dna(n, 100 + i, "ACGTN")) for i, n in enumerate([9000, 400, 15000, 7000, 120])]
    path = tmp_path / "multi.fa"
    write_fasta(str(path), recs)
    raw = open(path, "rb").read()
    whole = dg.pred.predict_fasta_tsv(w, raw, "f.fa", 50, 256, True, 50, 50)
    for world in (2, 3):
        pieces = [dg.pred.predict_fasta_tsv_sharded(w, raw, "f.fa", 50, 256, True, 50, 50, r, world)
                  for r in range(world)]
        owners = sharding.assign_records([len(s) for _, s in recs], world)
        for r in range(world):
            assert {k for k, _ in pieces[r]} <= {i for i, o in enumerate(owners) if o == r}
        assert sharding.merge_record_texts(pieces).decode() == whole


def test_position_sharding_then_finish_equals_whole_record(dg):
    from deepgrp_b200 import sharding
    T, U = 150, 32
    w = dg.model.random_weights(T, U, attention=True, seed=0).scaled(4.0)
    text = "NN" + random_dna(30_000, 77) + "N"
    labels, startpos, rows = dg.pred.predict_sequence(w, text.encode(), 50, 256, True, 50, 50)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    codes = fwd.argmax(axis=0).astype(np.uint8)
    L = codes.size
    parts = [sharding.predict_range(w, codes, L, a, b, 50, 256) for a, b in sharding.split_positions(L, 3)]
    lab = np.concatenate([p[0] for p in parts])
    sc = np.concatenate([p[1] for p in parts])
    out, rows2 = sharding.finish_record(lab, sc, 5, True, 50, 50, st)
    assert np.array_equal(out, labels)
    assert np.array_equal(rows2, rows)


def test_cli_end_to_end_with_hdf5_model(dg, oracle, tmp_path, capsys):
    """`deepgrp predict model.hdf5 a.fa b.fa --output out.tsv` and the README form without the
    sub-command; fused route vs the reference's five stepwise calls."""
    import sys
    from deepgrp_b200 import hdf5
    from deepgrp_b200.__main__ import CommandLineParser
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    mpath = str(tmp_path / "model.hdf5")
    hdf5.save_keras_model(mpath, w)
    fa1, fa2 = str(tmp_path / "a.fa"), str(tmp_path / "b.fa")
    write_fasta(fa1, [("one", "NN" + random_dna(8000, 1, "ACGTacgtN")), ("two", random_dna(3000, 2))])
    write_fasta(fa2, [("three", random_dna(5000, 3))])
    out1, out2 = str(tmp_path / "o1.tsv"), str(tmp_path / "o2.tsv")
    CommandLineParser().parse_args(["predict", mpath, fa1, fa2, "--output", out1]).set_logging().run()
    CommandLineParser().parse_args(["-s", "50", "predict", mpath, fa1, fa2, "--output", out2, "--stepwise"]).run()
    a, b = open(out1).read(), open(out2).read()
    assert a == b and a.count("\n") > 10
    assert a.splitlines()[0].split("\t")[:2] == [fa1, "one"]
    import gzip, shutil
    with open(fa1, "rb") as fi, gzip.open(fa1 + ".gz", "wb") as fo:   # gz input (SURVEY.md section 8f rank 2)
        shutil.copyfileobj(fi, fo)
    out3 = str(tmp_path / "o3.tsv")
    CommandLineParser().parse_args(["predict", mpath, fa1 + ".gz", "--output", out3]).run()
    assert open(out3).read().replace(fa1 + ".gz", fa1) == "".join(l + "\n" for l in a.splitlines() if l.startswith(fa1 + "\t"))
    CommandLineParser().parse_args([mpath, fa2]).run()            # README form, stdout
    assert capsys.readouterr().out == "".join(l + "\n" for l in a.splitlines() if l.startswith(fa2))


# ------------------------------------------------------------------ evaluation helpers
@pytest.mark.gpu
@pytest.mark.parametrize("min_len", (10, 20))
def test_filter_segments_reference_vector(dg, min_len):
    """tests/test_prediction.py:183-195 of the reference, through the GPU kernel."""
    segment_length = min_len * 2
    data = np.zeros(1000)
    data[110:110 + segment_length] = 1
    data[210 + segment_length:210 + 2 * segment_length] = 1
    expected = data.copy()
    data[0:min_len - 1] = 1
    data[120 + segment_length:120 + segment_length + min_len - 1] = 1
    data[(-min_len) + 1:] = 1
    dg.pred.filter_segments(data, min_len=min_len)
    np.testing.assert_equal(data, expected)


@pytest.mark.gpu
@pytest.mark.parametrize("n,min_len,seed", [(1, 1, 0), (7, 3, 1), (5000, 50, 2), (200_000, 50, 3), (200_000, 7, 4)])
def test_filter_segments_vs_oracle(dg, oracle, n, min_len, seed):
    rng = np.random.default_rng(seed)
    # runs of random length 1..2*min_len with labels 0..4, adjacent runs may share or change label
    lab = np.repeat(rng.integers(0, 5, size=n), rng.integers(1, 2 * min_len + 1, size=n))[:n].astype(np.int64)
    exp = lab.copy()
    oracle.filter_segments(exp, min_len)
    got = lab.copy()
    dg.pred.filter_segments(got, min_len)
    assert np.array_equal(got, exp)
    again = got.copy()
    dg.pred.filter_segments(again, min_len)       # idempotent
    assert np.array_equal(again, got)


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed", [(1, 0), (100, 1), (1_000_003, 2)])
def test_confusion_matrix_and_metrics_vs_oracle(dg, oracle, n, seed):
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 5, size=n)
    p = np.where(rng.random(n) < 0.7, t, rng.integers(0, 5, size=n))
    if n > 1:
        t[0], p[0] = 0, 4          # all five classes span the range
    else:
        t[:], p[:] = 0, 0          # a single label must be 0 (the matrix is 1 x 1, see the quirk test)
    exp = np.bincount(t * 5 + p, minlength=25).reshape(5, 5) if n > 1 else oracle.confusion_matrix(t, p)
    got = dg.pred.confusion_matrix(t, p)
    assert got.shape == exp.shape and np.array_equal(got, exp)
    if n == 100:
        assert np.array_equal(got, oracle.confusion_matrix(t, p))
    if n > 1:
        cnf, metrics = dg.pred.calculate_metrics(p, t)
        assert np.array_equal(cnf, exp)
        assert metrics["TotalACC"] == pytest.approx((t == p).mean())
        # MCC against the definition on the label vectors (multi-class R_K)
        s, c = n, float((t == p).sum())
        pk = np.bincount(p, minlength=5).astype(float)
        tk = np.bincount(t, minlength=5).astype(float)
        rk = (c * s - (pk * tk).sum()) / np.sqrt((s * s - (pk * pk).sum()) * (s * s - (tk * tk).sum()))
        assert metrics["MCC"] == pytest.approx(rk)
        assert metrics["TPR"].shape == (5,)


@pytest.mark.gpu
def test_confusion_matrix_reference_quirk(dg):
    """The reference sizes the matrix max - min + 1 and indexes with the raw labels, so labels that
    do not start at 0 raise IndexError there (prediction.py:212-217); same here."""
    with pytest.raises(IndexError):
        dg.pred.confusion_matrix(np.array([1, 2, 3]), np.array([1, 3, 2]))
