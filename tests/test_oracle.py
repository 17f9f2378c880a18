"""CPU tests of the oracle itself (the checker must be right before it checks anything):
* against golden vectors generated from the reference's own compiled natives
  (tests/golden/native_vectors.npz, made by tests/golden/make_golden.py);
* against the reference's known-answer tests, restated (reference tests/test_sequence.py,
  tests/test_mss.py, tests/test_prediction.py, tests/test_model.py:215-229);
* directly against oracle/_ref when it is present (the build container);
* forward numerics (parity unpinned in the reference): numpy float32 vs torch.nn.GRU vs float64.
"""
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(HERE, "golden", "native_vectors.npz"))


def test_oracle_encode_golden(oracle, golden):
    for i in range(int(golden["enc_n"])):
        text = golden["enc_text_%d" % i].tobytes()
        st, fwd = oracle.one_hot_encode_bytes(text)
        assert st == int(golden["enc_start_%d" % i])
        assert np.array_equal(fwd, golden["enc_fwd_%d" % i])


def test_oracle_get_max_golden(oracle, golden):
    for i in range(int(golden["max_n"])):
        out = oracle.get_max(golden["max_base_%d" % i].copy(), golden["max_in_%d" % i],
                             int(golden["max_stride_%d" % i]))
        assert np.array_equal(out, golden["max_out_%d" % i])


def test_oracle_segments_golden(oracle, golden):
    for i in range(int(golden["seg_n"])):
        got = oracle.yield_segments_array(golden["seg_lab_%d" % i], 11)
        assert np.array_equal(got, golden["seg_out_%d" % i])


def test_oracle_mss_golden(oracle, golden):
    for k in range(int(golden["mss_n"])):
        ml, xd = (int(v) for v in golden["mss_par_%d" % k])
        got = oracle.find_mss_relabel(golden["mss_s_%d" % k], golden["mss_lab_%d" % k], 5, ml, xd)
        assert np.array_equal(got, golden["mss_out_%d" % k]), k
        full = oracle.find_mss_labels(golden["mss_s_%d" % k], golden["mss_lab_%d" % k], 5, ml, xd)
        assert np.array_equal(full.argmax(axis=1), golden["mss_out_%d" % k])


def test_oracle_all_n_and_case(oracle):
    with pytest.raises(ValueError):
        oracle.one_hot_encode_dna_sequence("NNNN")
    st, fwd = oracle.one_hot_encode_dna_sequence("nnACGTnn")     # lowercase n is NOT trimmed
    assert st == 0 and fwd.shape == (5, 8) and fwd[4].tolist() == [1, 1, 0, 0, 0, 0, 1, 1]
    st, fwd = oracle.one_hot_encode_dna_sequence("")
    assert st == 0 and fwd.shape == (5, 0)


def test_oracle_segment_last_element_quirk(oracle):
    # SURVEY.md section 8a row a13: a run reaching the last element is split at size-1
    lab = np.array([0, 2, 2, 2, 2], np.int64)
    assert list(oracle.yield_segments(lab, 100)) == [(101, 104, 2), (104, 105, 2)]
    assert list(oracle.yield_segments(np.array([1, 0, 0], np.int64), 0)) == [(0, 1, 1), (2, 3, 0)]


def test_oracle_min_sc_truncation(oracle):
    # mss.c:35: `int min_sc` -- a 4.3-score segment passes min_mss_len=1 (threshold trunc(4.595)=4)
    s = np.array([-1.0, 4.3, -1.0])
    out = oracle.mss_find_all(s, np.log(99.0) * 1, -1.0)
    assert out.size == 1 and (out["st"][0], out["en"][0]) == (1, 2)
    out = oracle.mss_find_all(np.array([-1.0, 3.9, -1.0]), np.log(99.0) * 1, -1.0)
    assert out.size == 0


def test_oracle_score_transform_known_answer(oracle):
    # reference tests/test_prediction.py:39-64
    probs = np.array([[0.9, 0.1, 0, 0, 0], [0.1, 0.9, 0, 0, 0], [0.995, 0.005, 0, 0, 0],
                      [0, 0, 0, 0, 0]], dtype=np.float32)
    sc, cl = oracle.apply_mss_scores(probs)
    assert cl.tolist() == [0, 1, 0, 0]
    m = np.float32(0.9) + np.float32(1e-6)
    t = np.log(m / (1 - m))
    assert sc[0] == pytest.approx(-10 * t, rel=1e-6) and sc[1] == pytest.approx(t, rel=1e-6)
    assert sc[2] == pytest.approx(-10 * np.log(0.99 / 0.01), rel=1e-5)
    assert sc[3] == pytest.approx(138.155, abs=1e-2)            # never-covered row scores POSITIVE


def test_oracle_softmax_vs_scipy(oracle):
    from scipy.special import softmax as sp_softmax
    rng = np.random.default_rng(0)
    x = rng.random((100, 5)).astype(np.float32)
    assert np.allclose(oracle.softmax(x), sp_softmax(x, axis=1), atol=1e-6)


def test_oracle_windowing_and_partial_batch(oracle):
    # reference tests/test_prediction.py:16-36: ceil((L-T)/step) windows, short final batch
    L, T, step, B = 5000, 150, 50, 16
    fwd = np.zeros((5, L), np.int8)
    fwd[0] = 1
    batches = list(oracle.fetch_validation_batch(fwd, step, B, T))
    n_win = -(-(L - T) // step)
    assert sum(b.shape[0] for b in batches) == n_win == 97
    assert batches[-1].shape[0] == n_win % B == 1
    # prediction.py:105: the short batch lands at i * b_last * step
    pred = oracle.predict(lambda b: np.ones(b.shape[:2] + (5,), np.float32), iter(batches), (L, 5), step)
    covered = pred[:, 0] > 0
    assert covered[:(96 - 1) * step + T].all()
    assert not covered[(96 - 1) * step + T:].any()            # true tail window never placed


def test_oracle_reverse_complement_golden(oracle):
    # reference tests/test_model.py:215-229: reverse + channels [3,2,1,0,4]
    x = np.eye(5, dtype=np.float32)[[0, 1, 2, 3, 4, 0]][None]
    rc = oracle.reverse_complement(x)[0].argmax(axis=1)
    assert rc.tolist() == [3, 4, 0, 1, 2, 3]


def test_oracle_forward_engines_agree(oracle):
    from deepgrp_b200.model import random_weights
    for T, U, att in ((150, 32, True), (60, 60, True), (40, 16, False)):
        w = random_weights(T, U, attention=att, seed=1).as_dict()
        rng = np.random.default_rng(T)
        batch = np.eye(5, dtype=np.float32)[rng.integers(0, 5, size=(6, T))]
        a = oracle.model_forward(batch, w, dtype=np.float32, engine="numpy")
        b = oracle.model_forward(batch, w, dtype=np.float32, engine="torch")
        c = oracle.model_forward(batch, w, dtype=np.float64, engine="numpy")
        assert np.abs(a - c).max() < 5e-6 and np.abs(b - c).max() < 5e-6
        assert np.allclose(a.sum(axis=2), 1, atol=1e-5)


def test_oracle_fasta_reader(oracle, tmp_path):
    # reference tests/test_main.py:238-247 + the quirks of SURVEY.md section 8a row a1
    import io
    text = "ACGT\n>h1 desc\nacgt\nNNAC\n>\nGGGG\n>h3\nTT"
    recs = list(oracle.read_multi_fasta(io.StringIO(text)))
    assert recs == [("h1 desc", "ACGTNNAC"), ("h3", "TT")]
    with pytest.raises(IndexError):
        list(oracle.read_multi_fasta(io.StringIO(">a\nAC\n\nGT\n")))


def test_oracle_against_compiled_reference(oracle):
    """The oracle against the reference's natives on 40 seeded trials: live against oracle/_ref when it is built,
    otherwise against their outputs stored by tests/golden/make_golden.py (reference_trials.npz)."""
    import importlib.util
    from oracle import build_ref
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
    make_golden = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(make_golden)
    mods = build_ref.load()
    stored = os.path.join(HERE, "golden", "reference_trials.npz")
    if mods is not None:
        ref = make_golden.trial_vectors(*mods)
    elif os.path.exists(stored):
        ref = np.load(stored)
    else:
        pytest.skip("neither oracle/_ref nor tests/golden/reference_trials.npz (both come from the reference's "
                    "sources: python oracle/build_ref.py && python tests/golden/make_golden.py)")
    assert int(ref["n"]) == 40
    for i, (s, lab, text) in enumerate(make_golden.reference_trials()):
        for k, (ml, xd) in enumerate(make_golden.TRIAL_MSS_PARAMS):
            full = oracle.find_mss_labels(s, lab, 5, ml, xd)
            assert ((full == 0) | (full == 1)).all() and (full.sum(axis=1) == 1).all()
            assert np.array_equal(full.argmax(axis=1), ref["mss_%d_%d" % (i, k)]), (i, k)
        if set(text) != {"N"}:
            st, fwd = oracle.one_hot_encode_dna_sequence(text)
            assert st == int(ref["enc_start_%d" % i]) and np.array_equal(fwd, ref["enc_fwd_%d" % i]), i
        segs = np.array(list(oracle.yield_segments(lab, 5)), dtype=np.int64).reshape(-1, 3)
        assert np.array_equal(segs, ref["seg_%d" % i]), i


def test_oracle_lstm_engines_agree(oracle):
    from deepgrp_b200.model import random_weights
    w = random_weights(60, 24, attention=True, seed=1, rnn="LSTM").as_dict()
    rng = np.random.default_rng(0)
    batch = np.eye(5, dtype=np.float32)[rng.integers(0, 5, size=(4, 60))]
    a = oracle.model_forward(batch, w, engine="numpy")
    b = oracle.model_forward(batch, w, engine="torch")
    c = oracle.model_forward(batch, w, dtype=np.float64)
    assert np.abs(a - c).max() < 5e-6 and np.abs(b - c).max() < 5e-6


@pytest.mark.parametrize("min_len", (10, 20))
def test_oracle_filter_segments_reference_vector(oracle, min_len):
    """The known-answer case of the reference's tests/test_prediction.py:183-195."""
    segment_length = min_len * 2
    data = np.zeros(1000)
    data[110:110 + segment_length] = 1
    data[210 + segment_length:210 + 2 * segment_length] = 1
    expected = data.copy()
    data[0:min_len - 1] = 1
    data[120 + segment_length:120 + segment_length + min_len - 1] = 1
    data[(-min_len) + 1:] = 1
    oracle.filter_segments(data, min_len=min_len)
    np.testing.assert_equal(data, expected)


def test_oracle_confusion_matrix_vs_histogram(oracle):
    """tests/test_prediction.py:175-181 checks against pycm (absent here): same counts via bincount."""
    rng = np.random.default_rng(3)
    t = rng.integers(0, 4, size=100)
    p = rng.integers(0, 4, size=100)
    got = oracle.confusion_matrix(t, p)
    np.testing.assert_equal(got, np.bincount(t * 4 + p, minlength=16).reshape(4, 4))


# ---- pins for the floating-point half of the oracle (GRU / AdditiveAttention), beyond the two engines ---------
def test_gru_known_answer_by_hand():
    """A 2-unit, 3-step GRU with non-zero input AND recurrent biases, written out scalar by scalar from the Keras
    equations the reference's layer config selects (tests/test_model.json: reset_after=true, sigmoid / tanh;
    deepgrp/model.py:225-229): gate order z, r, h;  mx = x.W + b[0];  mh = h.R + b[1];
    z = sig(mx_z + mh_z);  r = sig(mx_r + mh_r);  hh = tanh(mx_h + r * mh_h);  h' = z h + (1 - z) hh.
    Step 1 from h = 0 with base A:  mx = (0.6, -0.45 | 0.175, 0.9 | -0.6, 0.45),  mh = b[1] = (-0.05, 0.1 | 0.2, -0.1 |
    0.15, -0.25);  z = sig(0.55), sig(-0.35);  r = sig(0.375), sig(0.8);  hh = tanh(-0.6 + r0 0.15), tanh(0.45 - r1 0.25);
    h1 = (1 - z) hh = (-0.172249633362514, 0.158736142330264).  The literals below were produced by exactly this
    scalar recipe (python floats, no matrix code) and pin both engines of the oracle."""
    from oracle import oracle as orc
    kernel = np.array([[0.5, -0.25, 0.125, 0.75, -0.5, 0.25], [0] * 6, [-0.75, 0.5, 0.25, -0.125, 0.375, -0.625],
                       [0.25, 0.25, -0.5, 0.5, 0.125, 0.875], [0] * 6], np.float64)
    rec = np.array([[0.5, -0.5, 0.25, 0.75, -0.25, 0.5], [-0.125, 0.375, 0.5, -0.25, 0.625, -0.375]], np.float64)
    bias = np.array([[0.1, -0.2, 0.05, 0.15, -0.1, 0.2], [-0.05, 0.1, 0.2, -0.1, 0.15, -0.25]], np.float64)
    # step 1 by hand, as in the docstring
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))
    z0, z1, r0, r1 = sig(0.55), sig(-0.35), sig(0.375), sig(0.8)
    h1 = [(1 - z0) * np.tanh(-0.6 + r0 * 0.15), (1 - z1) * np.tanh(0.45 - r1 * 0.25)]
    expected = np.array([[-0.17224963336251403, 0.15873614233026442],
                         [0.2437808425306526, -0.09622192184760324],
                         [0.16276491434039037, 0.3369773730450849]])
    assert np.allclose(h1, expected[0], rtol=0, atol=1e-15)
    x = np.eye(5)[[0, 2, 3]][None]                                    # bases A, G, T
    w = {"kernel": kernel, "recurrent_kernel": rec, "bias": bias}
    seq, last = orc.gru_sequence(x, w, dtype=np.float64)
    assert np.allclose(seq[0], expected, rtol=0, atol=1e-15) and np.allclose(last[0], expected[2], atol=1e-15)
    w32 = {k: v.astype(np.float32) for k, v in w.items()}
    seq_t, last_t = orc.gru_sequence_torch(x.astype(np.float32), w32)
    assert np.abs(seq_t[0] - expected).max() < 2e-7 and np.abs(last_t[0] - expected[2]).max() < 2e-7


def test_additive_attention_literal_broadcast_form():
    """Third, independently structured restatement of the attention block: Keras 2.5 AdditiveAttention
    ._calculate_scores literally -- reduce_sum(scale * tanh(q[:, :, None, :] + k[:, None, :, :]), -1) with
    q = reshape(hidden) [B, 1, U] and k = v = avg [B, T, U] -- then softmax over the value axis, matmul(weights, value),
    Flatten / RepeatVector / Concatenate([attention, avg]) / Dense / Softmax(axis=2) (deepgrp/model.py:311-329;
    layer configs in tests/test_model.json: use_scale=true, causal=false).  Must equal oracle.model_forward."""
    from oracle import oracle as orc
    import deepgrp_b200.model as dgmodel
    rng = np.random.default_rng(11)
    for T, U in ((7, 4), (23, 10)):
        w = dgmodel.random_weights(T, U, attention=True, seed=T).scaled(2.5).as_dict()
        w = {k: (v.astype(np.float64) if v is not None else None) for k, v in w.items()}
        w["bias"] = rng.normal(scale=0.3, size=w["bias"].shape)          # non-zero biases
        w["ff_bias"] = rng.normal(scale=0.3, size=w["ff_bias"].shape)
        x = np.eye(5)[rng.integers(0, 5, size=(3, T))]
        got = orc.model_forward(x, w, dtype=np.float64)
        fwd, hf = orc.gru_sequence(x, w, dtype=np.float64)
        rev, hr = orc.gru_sequence(orc.reverse_complement(x), w, dtype=np.float64)
        hidden = ((hf + hr) / 2).reshape(3, 1, U)                        # Average + Reshape((1, units))
        avg = (fwd + rev) / 2                                            # Average
        q, k, v = hidden, avg, avg
        q_r, k_r = q[:, :, None, :], k[:, None, :, :]                    # [B, Tq, 1, U], [B, 1, Tv, U]
        scores = np.sum(w["att_scale"] * np.tanh(q_r + k_r), axis=-1)    # [B, Tq = 1, Tv]
        e = np.exp(scores - scores.max(axis=-1, keepdims=True))
        weights = e / e.sum(axis=-1, keepdims=True)
        ctx = np.matmul(weights, v)                                      # [B, 1, U]
        rep = np.repeat(ctx.reshape(3, U)[:, None, :], T, axis=1)        # Flatten + RepeatVector(T)
        feat = np.concatenate([rep, avg], axis=-1)                       # Concatenate([attention, avg])
        logits = feat @ w["ff_kernel"] + w["ff_bias"]
        el = np.exp(logits - logits.max(axis=2, keepdims=True))
        exp = el / el.sum(axis=2, keepdims=True)
        assert np.abs(got - exp).max() < 1e-13, (T, U)
        # the torch-engine route (what the GPU parity tests compare against) agrees in float32
        w32 = {kk: (vv.astype(np.float32) if vv is not None else None) for kk, vv in w.items()}
        got32 = orc.model_forward(x.astype(np.float32), w32, engine="torch")
        assert np.abs(got32 - exp).max() < 5e-6, (T, U)
