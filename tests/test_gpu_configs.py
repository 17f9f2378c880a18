"""BASELINE.json configurations as parity cases.

config 1 (tests/test_model.json model T=150, U=32, 1 Mbp) is checked in full against the oracle;
the larger configurations are checked through size-independent properties (sharded == whole,
lower-case invariance, MSS only fills gaps, segments sorted/disjoint/consistent with labels, TSV row
count, idempotence of the label -> segments -> labels round trip)."""
import os

import numpy as np
import pytest

from conftest import random_dna, write_fasta

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dg(gpu_ctx):
    import deepgrp_b200.model as model
    import deepgrp_b200.prediction as pred
    import deepgrp_b200.sequence as seq
    import deepgrp_b200.sharding as sharding

    class NS:
        pass
    ns = NS()
    ns.model, ns.pred, ns.seq, ns.sharding, ns.ctx = model, pred, seq, sharding, gpu_ctx
    return ns


def synth(n, seed):
    rng = np.random.default_rng(seed)
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].tobytes()


def segments_to_labels(rows, length, startpos):
    lab = np.zeros(length, np.uint8)
    for s, e, l in zip(rows["start"], rows["end"], rows["label"]):
        lab[s - startpos:e - startpos] = l
    return lab


def check_rows_consistent(rows, labels, startpos):
    """rows are sorted, disjoint, label > 0, and paint exactly the non-zero labels."""
    assert (rows["label"] > 0).all()
    assert (rows["end"] > rows["start"]).all()
    assert (rows["start"][1:] >= rows["end"][:-1]).all()
    assert np.array_equal(segments_to_labels(rows, labels.size, startpos), labels)


def test_config1_full_parity(dg, oracle):
    """config 1: 1 Mbp, T=150, U=32, attention, step 50, batch 256 (W = 19 997, last batch 29):
    probabilities within 1e-3 (north_star), labels >= 99.99 % identical, startpos, TSV rows."""
    T, U, L = 150, 32, 1_000_000
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    raw = synth(L, 1)
    text = raw.decode()
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    got = dg.pred.predict(w, ds, (L, 5), 50)
    wd = w.as_dict()
    exp = oracle.predict(lambda b: oracle.model_forward(b, wd, engine="torch"),
                         oracle.fetch_validation_batch(fwd, 50, 256, T), (L, 5), 50)
    assert np.abs(got - exp).max() < 1e-3
    assert np.abs(got - exp).max() < 5e-6          # what the fp32-faithful kernel actually achieves
    assert np.array_equal(got == 0, exp == 0)      # same coverage incl. the displaced last batch of 29
    lab_g, lab_o = got.argmax(axis=1), exp.argmax(axis=1)
    assert (lab_g == lab_o).mean() >= 0.9999
    # MSS bit-exact given identical scores: feed the GPU's probabilities to the oracle's apply_mss
    from deepgrp_b200.model import Options
    mss_g = dg.pred.apply_mss(got, Options()).argmax(axis=1)
    sc, cl = dg.pred.mss_scores(got)
    mss_o = oracle.find_mss_relabel(sc, cl, 5, 50, 50)
    assert np.array_equal(mss_g, mss_o)
    labels, startpos, rows = dg.pred.predict_sequence(w, raw, 50, 256, True, 50, 50)
    assert startpos == 0 and np.array_equal(labels, mss_g)
    exp_rows = [(s, e, l) for s, e, l in oracle.yield_segments(mss_o.astype(np.int64), 0) if l > 0]
    assert list(zip(rows["start"].tolist(), rows["end"].tolist(), rows["label"].tolist())) == exp_rows


@pytest.mark.parametrize("scale", [1.0, 4.0])
def test_config2_shape_properties(dg, scale):
    """defaults.toml architecture (T=342, U=60) on a 5 Mbp record: position-sharded == whole (bitwise),
    MSS only fills gaps, rows consistent with labels, row extraction idempotent."""
    T, U, L = 342, 60, 5_000_000
    w = dg.model.random_weights(T, U, attention=True, seed=0).scaled(scale)
    raw = synth(L, 2)
    labels, startpos, rows = dg.pred.predict_sequence(w, raw, 50, 256, True, 50, 50)
    assert labels.size == L and startpos == 0
    check_rows_consistent(rows, labels, startpos)
    labels_nomss, _, rows_nomss = dg.pred.predict_sequence(w, raw, 50, 256, False, 50, 50)
    changed = labels != labels_nomss
    # gap fill never rewrites a non-zero label.  The only other differences are positions whose top
    # two probabilities are a few ulp apart: the no-MSS branch takes argmax AFTER the reference's
    # softmax (prediction.py:62-65), which can round them into a tie (first index wins), while
    # apply_mss takes argmax of the raw probabilities (prediction.py:51) -- reference behaviour.
    odd = changed & (labels_nomss != 0)
    assert odd.sum() <= 1e-5 * L
    assert (labels[changed & ~odd] > 0).all()
    codes = (np.frombuffer(raw, np.uint8) >> 1) & 3  # A=0 C=1 G=3 T=2 -> remap
    lut = np.zeros(256, np.uint8); lut[ord("A")] = 0; lut[ord("C")] = 1; lut[ord("G")] = 2; lut[ord("T")] = 3
    codes = lut[np.frombuffer(raw, np.uint8)]
    parts = [dg.sharding.predict_range(w, codes, L, a, b, 50, 256) for a, b in dg.sharding.split_positions(L, 4)]
    lab = np.concatenate([p[0] for p in parts]); sc = np.concatenate([p[1] for p in parts])
    out, rows2 = dg.sharding.finish_record(lab, sc, 5, True, 50, 50, 0)
    assert np.array_equal(out, labels) and np.array_equal(rows2, rows)
    # the never-covered tail (exclusive window range + displaced last batch) is class 0 before MSS
    n_win = len(range(0, L - T, 50))
    assert n_win % 256 != 0
    assert (labels_nomss[(n_win - 1) * 50 + T:] == 0).all()


def test_config4_shape_multirecord_softmask_and_n_runs(dg, tmp_path):
    """24 records with leading/trailing N runs, internal N runs and soft-masked lower case:
    lower case must not change anything; edge N is trimmed with a startpos offset; internal N is a
    fifth channel; contig sharding over 8 ranks merges to the single-rank text."""
    T, U = 342, 60
    w = dg.model.random_weights(T, U, attention=True, seed=0).scaled(4.0)
    rng = np.random.default_rng(4)
    recs_upper, recs_soft = [], []
    for k in range(24):
        n = int(rng.integers(20_000, 120_000))
        body = bytearray(synth(n, [4, k]))
        for _ in range(3):                                   # internal N runs
            a = int(rng.integers(0, n - 2000)); body[a:a + int(rng.integers(50, 1500))] = b"N" * 1
        i = int(rng.integers(1000, n - 6000))
        body[i:i + 5000] = b"N" * 5000
        seq = b"N" * int(rng.integers(1, 3000)) + bytes(body) + b"N" * int(rng.integers(1, 3000))
        soft = bytearray(seq)
        pos = 0
        while pos < len(soft):                               # lower-case runs, geometric lengths
            run = int(rng.geometric(1 / 300))
            if rng.random() < 0.5:
                soft[pos:pos + run] = bytes(soft[pos:pos + run]).lower()
            pos += run
        recs_upper.append(("chr%d some description" % (k + 1), seq.decode()))
        recs_soft.append(("chr%d some description" % (k + 1), bytes(soft).decode()))
    pu, ps = tmp_path / "upper.fa", tmp_path / "soft.fa"
    write_fasta(str(pu), recs_upper)
    write_fasta(str(ps), recs_soft)
    tsv_u = dg.pred.predict_fasta_tsv(w, open(pu, "rb").read(), "g.fa", 50, 256, True, 50, 50)
    tsv_s = dg.pred.predict_fasta_tsv(w, open(ps, "rb").read(), "g.fa", 50, 256, True, 50, 50)
    assert tsv_u == tsv_s and len(tsv_u) > 1000
    rows, records = dg.pred.predict_fasta(w, open(ps, "rb").read(), 50, 256, True, 50, 50)
    for (hdr, startpos, length), (h0, seq) in zip(records, recs_upper):
        assert hdr == h0
        assert startpos == len(seq) - len(seq.lstrip("N"))
        assert length == len(seq.strip("N"))
    assert (rows["start"] >= np.array([records[r][1] for r in rows["record"]])).all()
    raw = open(ps, "rb").read()
    pieces = [dg.pred.predict_fasta_tsv_sharded(w, raw, "g.fa", 50, 256, True, 50, 50, r, 8) for r in range(8)]
    assert dg.sharding.merge_record_texts(pieces).decode() == tsv_s


def test_config5_search_space_points(dg, oracle):
    """5a (T=260, U=50: the two-tile tcgen05 kernel) and 5b (T=512, U=128: the CTA-pair tcgen05 kernel,
    forward_tcw.cu), plus a width in between (U=90 pads to 128), against the oracle on a short record."""
    for (T, U, used_tc) in ((260, 50, 1), (512, 128, 3), (200, 90, 3)):
        w = dg.model.random_weights(T, U, attention=True, seed=5).scaled(3.0)
        text = random_dna(6000, T + U)
        st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
        ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
        got = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
        assert dg.ctx.get_int("forward_used_tc") == used_tc
        wd = w.as_dict()
        exp = oracle.predict(lambda b: oracle.model_forward(b, wd, engine="torch"),
                             oracle.fetch_validation_batch(fwd, 50, 256, T), (fwd.shape[1], 5), 50)
        assert np.abs(got - exp).max() < 2e-5
        assert (got.argmax(axis=1) == exp.argmax(axis=1)).mean() >= 0.9999


@pytest.mark.parametrize("wide,T,U,att", [(1, 150, 32, True), (1, 342, 60, True), (2, 342, 60, True),
                                           (2, 150, 40, False), (1, 100, 60, False)])
def test_wide_kernel_variants_match_the_two_tile_kernel(dg, oracle, wide, T, U, att):
    """forward_tcw.cu forced (forward_wide = 1: one CTA per tile, 2: CTA pair with tcgen05.mma.cta_group::2) on
    shapes the two-tile kernel also serves: both against the oracle and against each other."""
    w = dg.model.random_weights(T, U, attention=att, seed=21).scaled(3.0)
    text = random_dna(9_000 + 13 * T, T + U + wide)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    ref = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
    assert dg.ctx.get_int("forward_used_tc") == 1
    dg.ctx.set_int("forward_wide", wide)
    try:
        got = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
        used = dg.ctx.get_int("forward_used_tc")
    finally:
        dg.ctx.set_int("forward_wide", 0)
    assert used == 1 + wide
    assert np.abs(got - ref).max() < 2e-6
    wd = w.as_dict()
    exp = oracle.predict(lambda b: oracle.model_forward(b, wd, engine="torch"),
                         oracle.fetch_validation_batch(fwd, 50, 256, T), (fwd.shape[1], 5), 50)
    assert np.abs(got - exp).max() < 2e-5
    assert (got.argmax(axis=1) == exp.argmax(axis=1)).mean() >= 0.9999


@pytest.mark.parametrize("T,U,wide", [(200, 128, 0), (120, 100, 0), (150, 60, 1), (150, 60, 2)])
def test_wide_kernel_shapes_match_oracle(dg, oracle, T, U, wide):
    """The wide kernel against the oracle: at 100 and 128 units (CTA pair, two column blocks whose MMAs are
    issued block by block under the gate work) and forced at 60 units (one CTA or a CTA pair, one column
    block and one round of MMAs between two steps)."""
    w = dg.model.random_weights(T, U, attention=True, seed=31).scaled(3.0)
    text = random_dna(9_000 + 20 * T, T + U)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    dg.ctx.set_int("forward_wide", wide)
    try:
        got = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
        assert dg.ctx.get_int("forward_used_tc") == (3 if U > 64 else 1 + wide)
    finally:
        dg.ctx.set_int("forward_wide", 0)
    wd = w.as_dict()
    exp = oracle.predict(lambda b: oracle.model_forward(b, wd, engine="torch"),
                         oracle.fetch_validation_batch(fwd, 50, 256, T), (fwd.shape[1], 5), 50)
    assert np.abs(got - exp).max() < 2e-5
    assert (got.argmax(axis=1) == exp.argmax(axis=1)).mean() >= 0.9999


@pytest.mark.parametrize("key", ["forward_sum16", "forward_fp16x2", "forward_ub", "forward_overlap"])
def test_removed_forward_options_are_refused(dg, key):
    """Options that selected removed forward variants are unknown keys: a stale DEEPGRP_KNOBS setting fails
    instead of being ignored."""
    from deepgrp_b200._lib import DeepgrpError
    with pytest.raises(DeepgrpError, match="unknown option " + key):
        dg.ctx.set_int(key, 1)
    with pytest.raises(DeepgrpError, match="unknown option " + key):
        dg.ctx.get_int(key)


def test_window_slabs_compose(dg):
    """The window-probability buffer is bounded (forward_slab_mb): a record run in many small slabs gives the
    bit-identical prediction, including the displaced last batch (prediction.py:105)."""
    T, U = 150, 32
    w = dg.model.random_weights(T, U, attention=True, seed=3).scaled(4.0)
    text = random_dna(700_000, 77)
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    ref = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
    mb = dg.ctx.get_int("forward_slab_mb")
    dg.ctx.set_int("forward_slab_mb", 1)   # 4096-window slabs (the minimum)
    dg.ctx.set_int("forward_smem_vote", 0)  # the route with the window probabilities in HBM
    try:
        got = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
        dg.ctx.set_int("forward_slab_mb", mb)
        one = dg.pred.predict(w, ds, (fwd.shape[1], 5), 50)
    finally:
        dg.ctx.set_int("forward_slab_mb", mb)
        dg.ctx.set_int("forward_smem_vote", 1)
    assert np.array_equal(got, ref) and np.array_equal(one, ref)   # ref: the shared-memory vote (default)


def test_no_attention_model_through_the_fused_path(dg, oracle):
    """Options.attention=False (the class default, reference deepgrp/model.py:121, :321-323)."""
    w = dg.model.random_weights(150, 32, attention=False, seed=9).scaled(4.0)
    text = "N" + random_dna(20_000, 12) + "NN"
    labels, startpos, rows = dg.pred.predict_sequence(w, text.encode(), 50, 256, True, 50, 50)
    lab_o, st_o = oracle.predict_record(text, w.as_dict(), 150, 256, 50, True, engine="torch")
    assert startpos == st_o == 1
    assert (labels == lab_o).mean() >= 0.9999
    check_rows_consistent(rows, labels, startpos)


@pytest.mark.parametrize("T,U", [(150, 32), (90, 60), (40, 20)])
def test_lstm_variant(dg, oracle, tmp_path, T, U):
    """Options.rnn = "LSTM" (reference deepgrp/model.py:219-223): gates i, f, c, o, no attention."""
    from deepgrp_b200 import hdf5
    w = dg.model.random_weights(T, U, attention=True, seed=11, rnn="LSTM").scaled(2.0)
    assert w.att_scale is None and w.kernel.shape == (5, 4 * U)
    rng = np.random.default_rng(T)
    batch = np.eye(5, dtype=np.float32)[rng.integers(0, 5, size=(40, T))]
    got = w.predict_on_batch(batch)
    exp = oracle.model_forward(batch, w.as_dict())
    assert np.abs(got - exp).max() < 2e-5
    text = "NN" + random_dna(15_000, U) + "N"
    labels, startpos, rows = dg.pred.predict_sequence(w, text.encode(), 50, 256, True, 50, 50)
    assert dg.ctx.get_int("forward_used_tc") == 2   # the wide tcgen05 kernel, one CTA per tile
    lab_o, st_o = oracle.predict_record(text, w.as_dict(), T, 256, 50, True, engine="torch")
    assert startpos == st_o and (labels == lab_o).mean() >= 0.9999
    check_rows_consistent(rows, labels, startpos)
    path = str(tmp_path / "lstm.hdf5")
    hdf5.save_keras_model(path, w)
    w2 = dg.model.load_model(path)
    assert w2.rnn == "LSTM" and np.array_equal(w2.recurrent_kernel, w.recurrent_kernel)
    labels2, _, _ = dg.pred.predict_sequence(w2, text.encode(), 50, 256, True, 50, 50)
    assert np.array_equal(labels, labels2)


@pytest.mark.gpu
def test_chunk_sharding_device_entry_points(dg):
    """bench.py --shard chunk on one GPU: three position ranges through dgrp_predict_range_dev, concatenated
    on the device and finished with dgrp_finish_record_dev, give the row count of the whole-record call
    (and the same labels/scores as the host-pointer dgrp_predict_range)."""
    import ctypes
    import torch
    from deepgrp_b200 import _lib, sharding
    ctx = dg.ctx
    T, U, L = 150, 32, 61_234
    w = dg.model.random_weights(T, U, attention=True, seed=3).scaled(4.0)
    h = w.device_handle(ctx)
    codes = np.random.default_rng(5).integers(0, 4, size=L, dtype=np.uint8)
    d_codes = torch.from_numpy(codes).cuda()
    lib = _lib.lib()
    n_whole = ctypes.c_int64(0)
    _lib.check(lib.dgrp_predict_codes_dev(ctx.handle, h, ctypes.c_void_p(d_codes.data_ptr()), L, 50, 256, 1, 50, 50,
                                          _lib.COMPAT_REFERENCE, ctypes.byref(n_whole)))
    whole_lab = np.empty(L, dtype=np.uint8)
    whole_rows = np.empty((n_whole.value, 3), dtype=np.int64)
    _lib.check(lib.dgrp_predict_codes_dev_results(ctx.handle, _lib.ptr(whole_lab), L, _lib.ptr(whole_rows),
                                                  n_whole.value))
    full_lab = torch.empty(L, dtype=torch.uint8, device="cuda")
    full_sc = torch.empty(L, dtype=torch.float32, device="cuda")
    for (a, b) in sharding.split_positions(L, 3):
        lab = torch.empty(b - a, dtype=torch.uint8, device="cuda")
        sc = torch.empty(b - a, dtype=torch.float32, device="cuda")
        _lib.check(lib.dgrp_predict_range_dev(ctx.handle, h, ctypes.c_void_p(d_codes.data_ptr()), 0, L, L, a, b, 50, 256,
                                              _lib.COMPAT_REFERENCE, ctypes.c_void_p(lab.data_ptr()),
                                              ctypes.c_void_p(sc.data_ptr())))
        ctx.synchronize()
        host_lab, host_sc = sharding.predict_range(w, codes, L, a, b, 50, 256)
        assert np.array_equal(lab.cpu().numpy(), host_lab)
        assert np.array_equal(sc.cpu().numpy(), host_sc)
        full_lab[a:b] = lab
        full_sc[a:b] = sc
    torch.cuda.synchronize()
    n_rows = ctypes.c_int64(0)
    _lib.check(lib.dgrp_finish_record_dev(ctx.handle, ctypes.c_void_p(full_lab.data_ptr()),
                                          ctypes.c_void_p(full_sc.data_ptr()), L, 5, 1, 50, 50, ctypes.byref(n_rows)))
    assert n_rows.value == n_whole.value and n_rows.value > 0
    with pytest.raises(_lib.DeepgrpError):      # dgrp_finish_record_dev has overwritten those results
        _lib.check(lib.dgrp_predict_codes_dev_results(ctx.handle, _lib.ptr(whole_lab), L, None, 0))
    out, rows = sharding.finish_record(full_lab.cpu().numpy(), full_sc.cpu().numpy(), 5, True, 50, 50, 0)
    assert rows.size == n_rows.value
    # what dgrp_predict_codes_dev left on the device (bench.py --dump-outputs) is the whole-record result
    assert np.array_equal(whole_lab, out)
    assert np.array_equal(whole_rows, np.stack([rows["start"], rows["end"], rows["label"]], axis=1))


def test_predict_complete_from_files_on_disk(dg, oracle, tmp_path):
    """The evaluation route of the reference (deepgrp/optimization.py:58-69 around prediction.py:114-141) fed
    from the formats on disk: a gzip FASTA turned into the .npz one-hot file (preprocess_sequence), a
    training log directory holding TensorFlow checkpoints (training.py:53-59), the edge-N cut, predict_complete
    with and without MSS, then confusion matrix and metrics -- against the oracle on the same arrays."""
    import gzip
    from deepgrp_b200 import preprocessing, tfckpt
    T, U, step = 150, 32, 50
    w = dg.model.random_weights(T, U, attention=True, seed=3).scaled(4.0)
    wd = w.as_dict()
    logdir = tmp_path / "log"
    logdir.mkdir()
    names = {"layer_with_weights-0/cell/kernel": "kernel", "layer_with_weights-0/cell/recurrent_kernel": "recurrent_kernel",
             "layer_with_weights-0/cell/bias": "bias", "layer_with_weights-1/scale": "att_scale",
             "layer_with_weights-2/kernel": "ff_kernel", "layer_with_weights-2/bias": "ff_bias"}
    for epoch, factor in (("01", 0.5), ("02", 1.0)):            # the latest checkpoint holds the weights
        tfckpt.write_bundle(str(logdir / epoch), {k + "/.ATTRIBUTES/VARIABLE_VALUE": wd[v] * np.float32(factor)
                                                  for k, v in names.items()})
    fasta = tmp_path / "chrT.fa.gz"
    seq = "N" * 40 + random_dna(14_000, 21, "ACGTN") + "N" * 25
    with gzip.open(fasta, "wb") as fh:
        fh.write((">chrT\n" + "\n".join(seq[i:i + 70] for i in range(0, len(seq), 70)) + "\n").encode())
    assert preprocessing.preprocess_sequence(str(fasta)) is True
    fwd, _ = preprocessing.load_onehot_npz(str(fasta) + ".npz")
    assert fwd.shape == (5, len(seq)) and fwd[4, :40].all() and fwd[4, -25:].all()
    rng = np.random.default_rng(4)
    truth = np.repeat(rng.integers(0, 5, size=400), rng.integers(20, 90, size=400))[:len(seq)]
    y = np.zeros((5, len(seq)), dtype=np.int8)
    y[truth, np.arange(len(seq))] = 1
    fwd_cut, y_cut = preprocessing.drop_start_end_n(fwd, y)
    data = preprocessing.Data(fwd_cut, y_cut)
    opts = dg.model.Options(vecsize=T, batch_size=256, min_mss_len=50, xdrop_len=50)
    probs_o = oracle.predict(lambda b: oracle.model_forward(b, wd), oracle.fetch_validation_batch(fwd_cut, step, 256, T),
                             y_cut.shape[::-1], step)
    got_sm = dg.pred.predict_complete(step, opts, logdir, data, use_mss=False)
    assert got_sm.shape == y_cut.shape[::-1]
    assert np.abs(got_sm - oracle.softmax(probs_o)).max() < 1e-3
    got = dg.pred.predict_complete(step, opts, logdir, data, use_mss=True)
    exp = oracle.apply_mss(probs_o, 50, 50)
    assert got.shape == exp.shape and (got.sum(axis=1) == 1).all()
    agree = float((got.argmax(axis=1) == exp.argmax(axis=1)).mean())
    assert agree >= 0.9999, agree
    true_cls = y_cut.argmax(axis=0)
    cnf = dg.pred.confusion_matrix(true_cls, got.argmax(axis=1))
    assert np.array_equal(cnf, oracle.confusion_matrix(true_cls, got.argmax(axis=1)))
    assert int(np.asarray(cnf).sum()) == true_cls.size


def _multi_fasta(tmp_path, n_rec=5, seed=3, with_n=True):
    rng = np.random.default_rng(seed)
    recs = []
    for k in range(n_rec):
        n = int(rng.integers(3_000, 40_000))
        seq = random_dna(n, 100 + k)
        if with_n:
            seq = "N" * int(rng.integers(0, 30)) + seq + "N" * int(rng.integers(0, 30))
        recs.append(("rec%d description %d" % (k, n), seq))
    p = tmp_path / "multi.fa"
    write_fasta(str(p), recs)
    return open(p, "rb").read()


def test_fasta_stream_equals_one_shot(dg, tmp_path):
    """dgrp_fasta_stream_* (pipelined: host header index, per-slice upload, text copied back in pieces on a second
    stream) writes byte for byte what the one-shot dgrp_predict_fasta_tsv returns; sharded streams partition it."""
    import io
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    raw = _multi_fasta(tmp_path)
    ref = bytes(dg.pred.predict_fasta_tsv_view(w, raw, "m.fa", 50, 256, True, 50, 50))
    out = io.BytesIO()
    stats = dg.pred.predict_fasta_tsv_stream(w, raw, "m.fa", out, 50, 256, True, 50, 50)
    assert out.getvalue() == ref and len(ref) > 1000
    assert stats["records"] == 5 and stats["rows"] == ref.count(b"\n")
    # pinned source memory takes the direct-upload route
    import torch
    pinned = torch.empty(len(raw), dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = np.frombuffer(raw, dtype=np.uint8)
    out2 = io.BytesIO()
    dg.pred.predict_fasta_tsv_stream(w, pinned.numpy(), "m.fa", out2, 50, 256, True, 50, 50)
    assert out2.getvalue() == ref
    # all records are below the slice minimum here: one slice, rank 0 owns it
    parts = []
    for r in range(3):
        o = io.BytesIO()
        dg.pred.predict_fasta_tsv_stream(w, raw, "m.fa", o, 50, 256, True, 50, 50, rank=r, world=3)
        parts.append(o.getvalue())
    assert b"".join(parts) == ref


def test_fasta_stream_slices_and_errors(dg, tmp_path):
    """Records above the 8 MiB slice minimum are cut into slices and shared largest-first; an error (blank line)
    surfaces after the text of the records before it."""
    import io
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    recs = [("big%d" % k, random_dna(9_000_000 + 1000 * k, 50 + k)) for k in range(3)]
    p = tmp_path / "big.fa"
    write_fasta(str(p), recs)
    raw = open(p, "rb").read()
    ref = bytes(dg.pred.predict_fasta_tsv_view(w, raw, "b.fa", 50, 256, True, 50, 50))
    pieces = {}
    for r in range(2):
        with dg.pred.FastaTsvStream(w, raw, "b.fa", 50, 256, True, 50, 50, rank=r, world=2) as st:
            for sl, od, nr, last, view in st:
                pieces.setdefault((sl, od), []).append(bytes(view))
    assert sorted(pieces) == [(0, 0), (1, 0), (2, 0)]
    assert b"".join(b"".join(pieces[k]) for k in sorted(pieces)) == ref
    bad = raw[:len(raw) // 2] + b"\n\n" + raw[len(raw) // 2:]
    out = io.BytesIO()
    with pytest.raises(IndexError):
        dg.pred.predict_fasta_tsv_stream(w, bad, "b.fa", out, 50, 256, True, 50, 50)
    first = ref[:ref.index(b"b.fa\tbig1\t")]
    assert out.getvalue() == first          # record 0's rows were written before the error


@pytest.mark.parametrize("scale", (1.0, 4.0))
def test_config2_shape_vs_oracle_1mbp(dg, oracle, scale):
    """defaults.toml architecture (T = 342, U = 60, attention) on a 1 Mbp record against the oracle (torch engine,
    float32), with the random-init weight set and with the x4 (confident-output) set: probabilities within 1e-3
    (north_star; measured ~1e-6), labels >= 99.99 % identical, before and after MSS."""
    T, U, L = 342, 60, 1_000_000
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    if scale != 1.0:
        w = w.scaled(scale)
    text = synth(L, 2).decode()
    st, fwd = dg.seq.one_hot_encode_dna_sequence(text)
    ds = dg.pred.fetch_validation_batch(fwd, 50, 256, T)
    got = dg.pred.predict(w, ds, (L, 5), 50)
    assert dg.ctx.get_int("forward_used_tc") == 1
    wd = w.as_dict()
    exp = oracle.predict(lambda b: oracle.model_forward(b, wd, engine="torch"),
                         oracle.fetch_validation_batch(fwd, 50, 256, T), (L, 5), 50)
    dp = float(np.abs(got - exp).max())
    agree = float((got.argmax(axis=1) == exp.argmax(axis=1)).mean())
    print("config-2 shape, weights x%g: max |dp| %.3g, argmax agreement %.6f" % (scale, dp, agree))
    assert dp < (1e-5 if scale == 1.0 else 1e-4)
    assert agree >= 0.9999
    lab_g = dg.pred.apply_mss(got, dg.model.Options(min_mss_len=50, xdrop_len=50)).argmax(axis=1)
    lab_o = oracle.apply_mss(exp, 50, 50).argmax(axis=1)
    assert (lab_g == lab_o).mean() >= 0.9999


def test_config1_tsv_row_diff(dg, oracle, tmp_path):
    """BASELINE.json configs[0] end to end as text: the TSV the GPU pipeline writes for the 1 Mbp record against the
    oracle's restatement of the reference CLI, diffed row by row (tools/tsv_diff.py): the rows are the same up to
    the <= 1e-4 of the bases whose label sits on a near-tie of the probabilities."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import io
    import json
    import tsv_diff
    T, U, L = 150, 32, 1_000_000
    rows = {}
    for scale in (1.0, 4.0):
        w = dg.model.random_weights(T, U, attention=True, seed=0)
        if scale != 1.0:
            w = w.scaled(scale)
        p = tmp_path / "config1.fa"
        write_fasta(str(p), [("synthetic_1Mbp", synth(L, 1).decode())])
        out = io.BytesIO()
        dg.pred.predict_fasta_tsv_stream(w, open(p, "rb").read(), str(p), out, 50, 256, True, 50, 50)
        exp = oracle.predict_fasta_tsv(str(p), w.as_dict(), T, 256, 50, True, 50, 50, engine="torch")
        d = tsv_diff.diff_tsv(out.getvalue().decode(), exp)["total"]
        rows["weights_x%g" % scale] = d
        print("config 1, weights x%g:" % scale, json.dumps(d))
        assert d["rows_b"] > 1000
        assert d["bases_differ"] <= 1e-4 * L
        assert d["rows_only_a"] + d["rows_only_b"] <= 4 * max(1, d["bases_differ"])
    report = os.environ.get("DGRP_TSV_DIFF_REPORT")
    if report:
        json.dump({"workload": "BASELINE.json configs[0]: T=150, U=32, 1 Mbp, step 50, batch 256, MSS 50/50; "
                               "A = GPU pipeline (dgrp_fasta_stream), B = oracle restatement of the reference CLI",
                   "diff": rows}, open(report, "w"), indent=1)


@pytest.mark.parametrize("scale", (1.0, 4.0))
def test_vote_forms_agree_bit_for_bit(dg, scale):
    """The max-vote in its forms: (default) a tile's windows merged in shared memory and every row of the tile's span
    written once, shared rows by atomicMax; window probabilities in HBM + a gather pass fused with the score
    transform (label u8 + score f32 out, the float32[L, C] predictions never written); the same with a separate
    score kernel; the same with the windows in several slabs.  Same labels, same rows -- bit for bit, the vote
    being order-independent and the score transform the same instructions."""
    w = dg.model.random_weights(150, 32, attention=True, seed=5)
    if scale != 1.0:
        w = w.scaled(scale)
    text = ("NNN" + random_dna(400_000, 9) + "N").encode()
    out = {}
    try:
        # (shared-memory vote, fuse, slab MiB): the default; window probabilities in HBM + fused gather; the same
        # with a separate score pass; the same in several slabs
        for smem, fuse, slab_mb in ((1, 1, 8192), (0, 1, 8192), (0, 0, 8192), (0, 1, 1)):
            dg.ctx.set_int("forward_smem_vote", smem)
            dg.ctx.set_int("forward_fuse_score", fuse)
            dg.ctx.set_int("forward_slab_mb", slab_mb)
            labels, startpos, rows = dg.pred.predict_sequence(w, text, 50, 256, True, 50, 50)
            out[(smem, fuse, slab_mb)] = (labels.copy(), startpos, rows.copy(), dg.ctx.get_int("fused_last"))
    finally:
        dg.ctx.set_int("forward_smem_vote", 1)
        dg.ctx.set_int("forward_fuse_score", 1)
        dg.ctx.set_int("forward_slab_mb", 8192)
    assert [out[k][3] for k in ((1, 1, 8192), (0, 1, 8192), (0, 0, 8192), (0, 1, 1))] == [0, 1, 0, 0]   # "fused_last"
    ref = out[(0, 0, 8192)]
    for key, (labels, startpos, rows, _) in out.items():
        assert startpos == ref[1] and np.array_equal(labels, ref[0]) and np.array_equal(rows, ref[2]), key
    # a record shorter than the window: no window at all, every row scores +138.155 (class 0)
    short = dg.pred.predict_sequence(w, b"ACGTACGTAC" * 10, 50, 256, True, 50, 50)
    assert short[0].size == 100


def test_fasta_stream_can_be_abandoned(dg, tmp_path):
    """Closing a stream before it is exhausted (the caller broke out of its loop, or raised) stops the pipeline's
    threads without a hang and leaves the context usable."""
    import io
    import time
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    recs = [("r%d" % k, random_dna(9_000_000, 70 + k)) for k in range(3)]
    p = tmp_path / "three.fa"
    write_fasta(str(p), recs)
    raw = open(p, "rb").read()
    t0 = time.time()
    st = dg.pred.FastaTsvStream(w, raw, "t.fa", 50, 256, True, 50, 50)
    first = next(st)
    assert len(first[4]) > 0
    st.close()
    assert time.time() - t0 < 60
    out = io.BytesIO()
    stats = dg.pred.predict_fasta_tsv_stream(w, raw, "t.fa", out, 50, 256, True, 50, 50)   # the context still works
    assert stats["records"] == 3 and out.getvalue().count(b"\n") == stats["rows"]
