"""The options of `deepgrp predict` that change its output -- `-l/--min_mss_length`, `-x/--xdrop_length`,
`--no_use_mss`, `-s`, `-b` -- on every prediction route against the float64 oracle.

The other end-to-end tests run MSS with min_mss_len = xdrop_len = 50 only, where swapping the two lengths anywhere
along the wrappers and C entry points changes nothing, and the benchmark's scores take no x-drop reset at all.
Here the grid below runs through the device route at benchmark scale, the early-rows stream, chunk sharding and
synthetic score arrays whose x-drop resets sit where the chunked scan changes state (chunk, group and super-group
boundaries of `mss_chunk`), in the rounding regime of the running sum (|L| > 2^28) and with x-drop disabled.
Without MSS every route must give the labels of the reference's softmax over the record's global maximum, also
on a model whose top two classes are a few ulp apart."""
import ctypes
import io
import sys

import numpy as np
import pytest

from conftest import random_dna
from oracle import oracle as orc
from test_gpu_ranges import options
from test_gpu_scale import config2_codes, dg, onehot  # noqa: F401
from test_gpu_stream import early

# (min_mss_len, xdrop_len): the control; every candidate kept; threshold s0 * 7 truncated by (int) (mss.c:35);
# dense resets; x-drop disabled (xdrop_len <= 0 means -1, pymss.pyx:46-53); almost nothing kept
GRID = [(50, 50), (0, 50), (-5, 50), (7, 5), (50, 1), (1, 1), (50, 0), (50, -3), (500, 50)]
RESET_DENSE = {(50, 1), (1, 1)}
GRID_IDS = ["l%d_x%d" % g for g in GRID]
S0 = np.log(0.99 / (1 - 0.99))


def xdrop_of(xdrop_len):
    return S0 * xdrop_len * 10.0 if xdrop_len > 0 else -1.0


def rows_of(labels, startpos):
    """(start, end, label) rows of label > 0: yield_segments + the filter of __main__.py:288-290."""
    r = orc.yield_segments_array(np.asarray(labels, dtype=np.int64), startpos)
    return r[r[:, 2] > 0]


def tsv_of(filename, header, labels, startpos):
    return "".join("%s\t%s\t%d\t%d\t%d\n" % (filename, header, s, e, l)
                   for s, e, l in rows_of(labels, startpos)).encode()


def struct_rows(rows):
    return np.stack([rows["start"], rows["end"], rows["label"]], axis=1).astype(np.int64)


# ------------------------------------------------------------------ synthetic score regimes
CH = 512                    # mss_chunk of the synthetic tests: chunk k holds positions [k * CH, (k + 1) * CH)
GROUP, SUPER = 32 * CH, 1024 * CH
N_SYN = 46_800_000          # at least the benchmark record
RESET_DIP = {"boundaries": -100.0, "rounding": -5000.0}


def _sawtooth(rng, n, a, b):
    """Scores +a[k] at even positions and -b[k] at odd ones with b <= a: the running sum never falls below its
    value after the previous pair, so it stays within max(b) of its peak -- no x-drop reset fires on its own."""
    S = np.empty(n, dtype=np.float32)
    S[0::2] = a[:(n + 1) // 2]
    S[1::2] = -np.minimum(a, b)[:n // 2]
    return S


def synthetic_scores(regime):
    """(float32 scores[N_SYN], planned reset positions) of a seeded regime.

    * "boundaries": integer scores, a sawtooth of +1..40 / -1..40 (drawdown <= 40 < s0 * 10 = 45.9, the x-drop of
      xdrop_len 1) with a dip of -100 that resets at xdrop_len 1 (not at 50): in every fifth chunk at its last, first
      or second element (k * CH - 1, k * CH, k * CH + 1 in turn), and the same at every group (32 chunks) and
      super-group (1024 chunks) boundary.
    * "rounding": +30..50 / -0..1 float32 scores whose low bits reach 2^-24 and beyond: the running sum drifts up
      by ~20 per position, past 2^28 (where its double additions round), until a dip of -5000 resets it (at
      xdrop_len <= 108) mid super-group 34; it drifts past 2^28 again until the second dip mid super-group 78.
    * "downward": integer scores -3..3 of mean -0.16 without any dip: the stack is flushed at every new minimum,
      and an x-drop reset would fire everywhere (the running sum falls without bound below its peak), so this is the
      regime of x-drop disabled; its segments score small integers, thousands of them exactly the (int) threshold
      s0 * 7 -> 32."""
    if regime == "boundaries":
        rng = np.random.default_rng(101)
        h = (N_SYN + 1) // 2
        S = _sawtooth(rng, N_SYN, rng.integers(1, 41, h).astype(np.float32), rng.integers(1, 41, h).astype(np.float32))
        want = {k * CH + (k // 5 % 3) - 1 for k in range(5, N_SYN // CH, 5)}
        want |= {j * GROUP + (j % 3) - 1 for j in range(1, N_SYN // GROUP)}
        want |= {j * SUPER + (j % 3) - 1 for j in range(1, N_SYN // SUPER)}
        resets = []
        for p in sorted(want):            # a reset needs a positive run since the previous one
            if not resets or p - resets[-1] >= 3:
                resets.append(p)
    elif regime == "rounding":
        rng = np.random.default_rng(102)
        h = (N_SYN + 1) // 2
        S = _sawtooth(rng, N_SYN, rng.uniform(30, 50, h).astype(np.float32), rng.uniform(0, 1, h).astype(np.float32))
        resets = [34 * SUPER + 77, 78 * SUPER + 300]
    elif regime == "downward":
        rng = np.random.default_rng(103)
        S = rng.choice(np.array([-3, -2, -1, 1, 2, 3], np.float32), size=N_SYN, p=[0.15, 0.2, 0.17, 0.2, 0.18, 0.1])
        resets = []
    else:
        raise ValueError(regime)
    resets = np.array(resets, dtype=np.int64)
    if regime in RESET_DIP:
        S[resets] = RESET_DIP[regime]
    return S, resets


def synthetic_labels(S, seed):
    """Labels 1..4 where the score is positive and 0 elsewhere, as the score transform gives them."""
    rng = np.random.default_rng(seed)
    return np.where(S > 0, rng.integers(1, 5, S.size), 0).astype(np.uint8)


def reset_positions_hold(S, planned, xdrop):
    """True when, with the x-drop `xdrop`, the reference's scan (oracle_c.c:175-179: reset where a non-positive
    score takes the running sum more than xdrop below the highest run end since the last reset) resets at the
    `planned` positions and nowhere else.  Running sums by np.cumsum in float64."""
    G = np.cumsum(S.astype(np.float64))
    bounds = [0] + [int(p) for p in planned] + [S.size]
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        c = G[r0:r1] - (G[r0 - 1] if r0 > 0 else 0.0)      # after a reset at r0: cum = S[r0]
        pos = S[r0:r1] > 0
        peak = np.maximum.accumulate(np.where(pos, c, -np.inf))
        if xdrop > 0 and ((~pos[1:]) & (c[1:] + xdrop < peak[:-1])).any():
            return False                                    # a reset that was not planned
        if r1 < S.size and not (S[r1] <= 0 and xdrop > 0 and c[-1] + float(S[r1]) + xdrop < peak[-1]):
            return False                                    # a planned reset that does not fire
    return True


def test_synthetic_regimes_reach_their_targets():
    """Each generator reaches the regime its GPU test is about (checked with np.cumsum in float64)."""
    S, R = synthetic_scores("boundaries")
    assert S.size >= 46_700_000 and np.array_equal(S, np.round(S))
    assert reset_positions_hold(S, R, xdrop_of(1))          # resets exactly where planned
    assert reset_positions_hold(S, [], xdrop_of(50))        # and none at the default x-drop
    off = R % CH
    for o in (CH - 1, 0, 1):                                # last, first and second element of a chunk
        assert np.count_nonzero(off == o) > 1000
    for unit in (GROUP, SUPER):                             # at group and super-group boundaries
        near = np.abs(R - np.round(R / unit) * unit) <= 1
        assert np.count_nonzero(near & (R >= unit - 1)) >= N_SYN // unit - 1
    S, R = synthetic_scores("rounding")
    assert reset_positions_hold(S, R, xdrop_of(50)) and reset_positions_hold(S, R, xdrop_of(1))
    G = np.cumsum(S.astype(np.float64))
    before, between = G[:R[0]], G[R[0]:R[1]] - G[R[0] - 1]
    assert before.max() > 2 ** 28 and between.max() > 2 ** 28  # drift past 2^28, reset, drift past it again
    # the double additions round there: the increment of the running sum is not the score (np.diff is exact)
    high = np.abs(G[:-1]) > 2 ** 28
    assert np.count_nonzero((np.diff(G) != S[1:].astype(np.float64)) & high) > 1_000_000
    S, R = synthetic_scores("downward")
    G = np.cumsum(S.astype(np.float64))
    assert R.size == 0 and G[-1] < -5e6 and np.array_equal(S, np.round(S))
    new_min = np.flatnonzero(G < np.minimum.accumulate(np.concatenate([[0.0], G[:-1]])))
    assert new_min.size > 100_000                           # flushes all along the record
    assert (np.maximum.accumulate(G) - G).max() > xdrop_of(1) * 1000


# regime -> (min_mss_len, xdrop_len) cases; every case with x-drop on is checked against x-drop off
SYN_CASES = {
    "boundaries": [(50, 1), (0, 1), (7, 1), (500, 1), (50, 0), (7, 0)],
    "rounding": [(50, 50), (0, 50), (500, 50), (50, 1), (50, 0)],
    "downward": [(7, 0), (0, 0), (7, -3), (500, 0), (7, 1)],
}


@pytest.mark.gpu
@pytest.mark.parametrize("regime", list(SYN_CASES))
def test_finish_record_of_synthetic_regimes_equals_oracle(dg, oracle, regime):
    """dgrp_finish_record on 46.8 M float32 scores of a synthetic regime, chunks of 512: labels are the oracle's MSS
    relabelling and rows its segments, bit for bit, without the sequential completion; where resets fire, the
    result differs from the same scores with x-drop disabled (so the reset path ran)."""
    S, R = synthetic_scores(regime)
    lab = synthetic_labels(S, seed=len(regime))
    S64 = S.astype(np.float64)
    with options(dg.ctx, mss_chunk=CH):
        for mn, xd in SYN_CASES[regime]:
            out, rows = dg.sharding.finish_record(lab, S, 5, True, mn, xd, 0)
            rounds = dg.ctx.get_int("mss_rounds")
            exp = oracle.find_mss_relabel(S64, lab, 5, mn, xd)
            ok = np.array_equal(out, exp)
            er = rows_of(exp, 0)
            print("%s l=%d x=%d: %d MSS rounds, %d rows, %d positions relabelled%s"
                  % (regime, mn, xd, rounds, rows.size, np.count_nonzero(exp != lab), "" if ok else ", MISMATCH"))
            assert rounds > 0, (regime, mn, xd)
            assert ok, (regime, mn, xd, int(np.count_nonzero(out != exp)))
            assert np.array_equal(struct_rows(rows), er), (regime, mn, xd)
            if xd > 0:
                assert not np.array_equal(exp, oracle.find_mss_relabel(S64, lab, 5, mn, 0)), (regime, mn, xd)


# ------------------------------------------------------------------ A. the device route at benchmark scale
def codes_dev(ctx, h, d_codes, L, step, batch, use_mss, mn, xd):
    """dgrp_predict_codes_dev + _results: (labels, rows int64[n, 3], MSS rounds)."""
    from deepgrp_b200 import _lib
    lib = _lib.lib()
    n_rows = ctypes.c_int64(0)
    _lib.check(lib.dgrp_predict_codes_dev(ctx.handle, h, ctypes.c_void_p(d_codes.data_ptr()), L, step, batch,
                                          int(use_mss), mn, xd, _lib.COMPAT_REFERENCE, ctypes.byref(n_rows)))
    rounds = ctx.get_int("mss_rounds")
    labels = np.empty(L, dtype=np.uint8)
    rows = np.empty((n_rows.value, 3), dtype=np.int64)
    _lib.check(lib.dgrp_predict_codes_dev_results(ctx.handle, _lib.ptr(labels), L, _lib.ptr(rows), n_rows.value))
    return labels, rows, rounds


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 4.0])
def test_config2_device_route_with_the_options(dg, oracle, scale):
    """The benchmark's call on its record (46.7 Mbp, random-init weights x1 and x4) for every option pair: labels
    are the oracle's MSS of the GPU's own scores and rows its segments, bit for bit, without the sequential
    completion; the reset-dense pairs differ from x-drop disabled."""
    import torch
    T, U, step, batch = 342, 60, 50, 256
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    if scale != 1.0:
        w = w.scaled(scale)
    codes = config2_codes()
    L = codes.size
    probs = dg.pred.predict(w, dg.pred.fetch_validation_batch(onehot(codes), step, batch, T), (L, 5), step)
    sc, cl = dg.pred.mss_scores(probs)
    del probs
    h = w.device_handle(dg.ctx)
    d_codes = torch.from_numpy(codes).cuda()
    for mn, xd in GRID:
        labels, rows, rounds = codes_dev(dg.ctx, h, d_codes, L, step, batch, True, mn, xd)
        print("config 2 x%g, l=%d x=%d: %d MSS rounds, %d rows" % (scale, mn, xd, rounds, rows.shape[0]))
        assert rounds > 0, (mn, xd)
        exp = oracle.find_mss_relabel(sc, cl, 5, mn, xd)
        assert np.array_equal(labels, exp), (mn, xd, int(np.count_nonzero(labels != exp)))
        assert np.array_equal(rows, rows_of(exp, 0)), (mn, xd)
        if (mn, xd) in RESET_DENSE and scale == 4.0:
            # the x4 scores drift upwards and never flush on their own, so the resets show in the result; the x1
            # scores drift downwards and flush at every new minimum, which is where a reset would have cut anyway
            assert not np.array_equal(exp, oracle.find_mss_relabel(sc, cl, 5, mn, 0)), (mn, xd)
    del d_codes


# ------------------------------------------------------------------ B. the early-rows stream
def record(n, seed, n_runs=False, header="chrT"):
    """(FASTA bytes, sequence) of one record of n random bases; n_runs: N runs inside and at both ends."""
    seq = random_dna(n, seed)
    if n_runs:
        rng = np.random.default_rng(seed)
        s = list(seq)
        for _ in range(6):
            a, k = int(rng.integers(0, n - 500)), int(rng.integers(5, 400))
            s[a:a + k] = ["N"] * k
        seq = "NNNN" + "".join(s) + "NN"
    return (">" + header + "\n" + "\n".join(seq[i:i + 70] for i in range(0, len(seq), 70)) + "\n").encode(), seq


def gpu_probs(dg, oracle, w, seq, step, batch):
    """(startpos, float32 probabilities of the trimmed record, trimmed codes) on the GPU forward."""
    startpos, fwd = oracle.one_hot_encode_dna_sequence(seq)
    L = fwd.shape[1]
    probs = dg.pred.predict(w, dg.pred.fetch_validation_batch(fwd, step, batch, w.vecsize), (L, 5), step)
    return startpos, probs, fwd.argmax(axis=0).astype(np.uint8)


# name, T, U, weight scale, bases, seed, N runs, step, batch.  "bench_x4" is the benchmark's shape with the x4 weights:
# on it (not on the T = 150 ones) x-drop resets at xdrop_len 1 change the result
STREAM_CASES = [("x1", 150, 32, 1.0, 60_000, 7, False, 50, 256), ("x4", 150, 32, 4.0, 60_000, 7, False, 50, 256),
                ("nruns_s37_b7", 150, 32, 1.0, 41_234, 21, True, 37, 7),
                ("bench_x4", 342, 60, 4.0, 60_000, 7, False, 50, 256)]


@pytest.fixture(scope="module")
def stream_inputs(dg, oracle):
    """name -> (weights, FASTA bytes, startpos, MSS scores, classes, step, batch)."""
    out = {}
    for name, T, U, scale, n, seed, n_runs, step, batch in STREAM_CASES:
        w = dg.model.random_weights(T, U, attention=True, seed=0 if not n_runs else 3).scaled(scale)
        raw, seq = record(n, seed, n_runs)
        startpos, probs, _ = gpu_probs(dg, oracle, w, seq, step, batch)
        sc, cl = dg.pred.mss_scores(probs)
        out[name] = (w, raw, startpos, sc, cl, step, batch)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mn,xd", GRID, ids=GRID_IDS)
def test_early_rows_stream_with_the_options(dg, oracle, stream_inputs, mn, xd):
    """The early-rows stream in 2, 3 and 6 slabs gives the one-shot text byte for byte, and the one-shot text is
    the oracle's MSS of the GPU's probabilities.  In the reset-dense cases the resets change the result on the
    benchmark's shape with the x4 weights (its scores drift upwards and flush only where a reset clears the stack;
    its first slab flushes too little, so the stream finishes it as a whole), and rows of the x1 record leave
    early: the resumed scan runs with x-drop 1."""
    for name, (w, raw, startpos, sc, cl, step, batch) in stream_inputs.items():
        ref = bytes(dg.pred.predict_fasta_tsv_view(w, raw, "o.fa", step, batch, True, mn, xd))
        exp = oracle.find_mss_relabel(sc, cl, 5, mn, xd)
        assert ref == tsv_of("o.fa", "chrT", exp, startpos), (name, mn, xd)
        parts = []
        for slabs in (2, 3, 6):
            with early(dg.ctx, 2, 48, slabs):
                out = io.BytesIO()
                stats = dg.pred.predict_fasta_tsv_stream(w, raw, "o.fa", out, step, batch, True, mn, xd)
                parts.append(dg.ctx.get_int("stream_early_parts"))
            assert out.getvalue() == ref, (name, mn, xd, slabs)
            assert stats["rows"] == ref.count(b"\n")
        differs = int(np.count_nonzero(exp != oracle.find_mss_relabel(sc, cl, 5, mn, 0)))
        print("%s l=%d x=%d: %d rows, early parts %s, %d positions differ from x-drop off"
              % (name, mn, xd, ref.count(b"\n"), parts, differs))
        if (mn, xd) in RESET_DENSE and name == "bench_x4":
            assert differs > 0, name
        if (mn, xd) in RESET_DENSE and name == "x1":
            assert min(parts) >= 1, (name, parts)


# ------------------------------------------------------------------ C. chunk sharding
@pytest.mark.gpu
@pytest.mark.parametrize("mn,xd", GRID, ids=GRID_IDS)
def test_chunk_sharding_with_the_options(dg, oracle, stream_inputs, mn, xd):
    """3 and 8 position ranges through predict_range, then finish_record with the options, give predict_sequence's
    labels and rows."""
    for name, (w, raw, startpos, sc, cl, step, batch) in stream_inputs.items():
        seq = b"".join(raw.split(b"\n")[1:])
        labels, sp, rows = dg.pred.predict_sequence(w, seq, step, batch, True, mn, xd)
        assert sp == startpos
        assert np.array_equal(labels, oracle.find_mss_relabel(sc, cl, 5, mn, xd)), (name, mn, xd)
        _, fwd = oracle.one_hot_encode_dna_sequence(seq.decode())
        codes = fwd.argmax(axis=0).astype(np.uint8)
        L = codes.size
        for k in (3, 8):
            parts = [dg.sharding.predict_range(w, codes, L, a, b, step, batch)
                     for a, b in dg.sharding.split_positions(L, k)]
            out, rows2 = dg.sharding.finish_record(np.concatenate([p[0] for p in parts]),
                                                   np.concatenate([p[1] for p in parts]), 5, True, mn, xd, startpos)
            assert np.array_equal(out, labels), (name, k, mn, xd)
            assert np.array_equal(struct_rows(rows2), struct_rows(rows)), (name, k, mn, xd)


# ------------------------------------------------------------------ D. MSS off on every route
def near_tie_weights(dg, kind):
    """T = 150, U = 32 random-init weights; "near_tie": FF column 2 a copy of column 1, both biases + 2.0 so that
    classes 1 and 2 are on top, and class 2's bias the next float32 above class 1's; "exact_tie": equal biases."""
    w = dg.model.random_weights(150, 32, attention=True, seed=9)
    if kind in ("x1", "x4"):
        return w.scaled(4.0) if kind == "x4" else w
    fk, fb = w.ff_kernel.copy(), w.ff_bias.copy()
    fk[:, 2] = fk[:, 1]
    fb[1] += np.float32(2.0)
    fb[2] = np.nextafter(fb[1], np.float32(np.inf)) if kind == "near_tie" else fb[1]
    return dg.model.ModelWeights(w.vecsize, w.units, w.kernel, w.recurrent_kernel, w.bias, fk, fb, w.att_scale)


# The GPU's softmax (vote.cu softmax_rows_kernel) uses expf, within 2 ulp of exp (CUDA C Programming Guide, table
# of single-precision functions), where numpy rounds exp correctly: the top two softmax values of a row may each be
# 2 ulp off, so whether they tie (first index wins) can differ from the oracle up to 4 ulp apart; 6 with the
# division's rounding.
SM_ULPS = 6
NOMSS_RECORDS = [("chrA", 200_000, 41, False), ("chrB", 60_000, 42, True), ("chrC", 20_000, 43, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["near_tie", "exact_tie", "x1", "x4"])
def test_no_mss_on_every_route(dg, oracle, tmp_path, monkeypatch, kind):
    """Without MSS, predict_sequence (with either vote form), dgrp_predict_codes_dev, the one-shot TSV, the stream, contig sharding and the
    CLI (`--no_use_mss -l 7 -x 1`: the lengths are ignored) give bit-identical labels and rows, and the labels are
    the argmax of the oracle's softmax of the GPU's probabilities except where the top two probabilities are near
    a tie (within 2 ulp raw, or SM_ULPS ulp after the softmax).  Chunk sharding is refused without MSS: its labels (the ranges' argmax of the raw vote) differ from the
    whole record's exactly at such near-ties."""
    import torch
    from deepgrp_b200 import _lib, __main__ as cli
    w = near_tie_weights(dg, kind)
    step, batch = 50, 256
    raws, seqs = zip(*[record(n, seed, n_runs, header) for header, n, seed, n_runs in NOMSS_RECORDS])
    raw = b"".join(raws)
    fasta = tmp_path / "in.fa"
    fasta.write_bytes(raw)
    fname = str(fasta)
    exp_text, n_near, n_div = [], 0, 0
    for (header, _, _, _), seq in zip(NOMSS_RECORDS, seqs):
        startpos, probs, codes = gpu_probs(dg, oracle, w, seq, step, batch)
        L = codes.size
        labels, sp, rows = dg.pred.predict_sequence(w, seq.encode(), step, batch, False, 50, 50)
        labels2, _, rows2 = dg.pred.predict_sequence(w, seq.encode(), step, batch, False, 7, 1)
        assert sp == startpos and labels.size == L
        assert np.array_equal(labels, labels2) and np.array_equal(struct_rows(rows), struct_rows(rows2))
        # the vote form whose gather pass can fuse the score transform (argmax of the raw vote) when MSS is on
        with options(dg.ctx, forward_smem_vote=0):
            labels3, _, _ = dg.pred.predict_sequence(w, seq.encode(), step, batch, False, 50, 50)
        assert np.array_equal(labels, labels3)
        assert np.array_equal(struct_rows(rows), rows_of(labels, startpos))
        d_codes = torch.from_numpy(codes).cuda()
        lab_dev, rows_dev, _ = codes_dev(dg.ctx, w.device_handle(dg.ctx), d_codes, L, step, batch, False, 7, 1)
        del d_codes
        assert np.array_equal(lab_dev, labels) and np.array_equal(rows_dev, rows_of(labels, 0))
        # the oracle: argmax of the softmax over the record's global maximum (prediction.py:62-65).  Near-ties:
        # the top two probabilities within 2 ulp, or their softmax values within SM_ULPS ulp (exp(p - max) near 1
        # has a coarser grid than p itself, so raw probabilities a few ulp apart can round to one value there)
        sm = oracle.softmax(probs)
        ref = sm.argmax(axis=1)
        order = np.argsort(probs, axis=1, kind="stable")[:, -2:]
        rows_i = np.arange(L)[:, None]
        top2, sm2 = probs[rows_i, order], sm[rows_i, order]
        near = ((top2[:, 1] - top2[:, 0] <= 2 * np.spacing(top2[:, 1]))
                | (np.abs(sm2[:, 1] - sm2[:, 0]) <= SM_ULPS * np.spacing(sm2.max(axis=1))))
        off = labels != ref
        assert not (off & ~near).any(), (kind, header, np.flatnonzero(off & ~near)[:10])
        # chunk sharding: the ranges' labels are the raw vote's argmax
        rl = np.concatenate([dg.sharding.predict_range(w, codes, L, a, b, step, batch)[0]
                             for a, b in dg.sharding.split_positions(L, 8)])
        assert np.array_equal(rl, probs.argmax(axis=1))
        div = rl != labels
        assert not (div & ~near).any(), (kind, header)
        n_near += int(near.sum())
        n_div += int(div.sum())
        print("%s %s: %d bases, %d near-tie positions, %d of them off the oracle's softmax argmax, %d where the "
              "ranges' raw-vote labels differ from the whole record's" % (kind, header, L, near.sum(), off.sum(),
                                                                         div.sum()))
        exp_text.append(tsv_of(fname, header, labels, startpos))
        with pytest.raises(ValueError, match="use_mss"):
            dg.sharding.finish_record(rl, np.zeros(L, np.float32), 5, False, 50, 50, startpos)
    if kind == "near_tie":
        # 2 138 positions over the three records on a B200: chunk-sharded labels without MSS would differ there
        assert n_near > 1000 and n_div > 0
    if kind == "exact_tie":
        assert n_div == 0
    exp_text = b"".join(exp_text)
    assert exp_text.count(b"\n") >= len(NOMSS_RECORDS)
    one_shot = bytes(dg.pred.predict_fasta_tsv_view(w, raw, fname, step, batch, False, 7, 1))
    assert one_shot == exp_text
    out = io.BytesIO()
    dg.pred.predict_fasta_tsv_stream(w, raw, fname, out, step, batch, False, 7, 1)
    assert out.getvalue() == exp_text
    pieces = [dg.pred.predict_fasta_tsv_sharded(w, raw, fname, step, batch, False, 7, 1, r, 2) for r in range(2)]
    assert dg.sharding.merge_record_texts(pieces) == exp_text
    if kind == "near_tie":
        mpath, opath = str(tmp_path / "m.npz"), str(tmp_path / "out.tsv")
        w.save_npz(mpath)
        monkeypatch.setattr(sys, "argv", ["deepgrp", "-l", "7", "-x", "1", "predict", "--no_use_mss", mpath, fname,
                                          "--output", opath])
        cli.main()
        with open(opath, "rb") as fh:
            assert fh.read() == exp_text
    n_rows = ctypes.c_int64(0)
    assert _lib.lib().dgrp_finish_record(dg.ctx.handle, _lib.ptr(np.zeros(8, np.uint8)),
                                         _lib.ptr(np.zeros(8, np.float32)), 8, 5, 0, 50, 50, 0, None, None, 0,
                                         ctypes.byref(n_rows)) == _lib.E_UNSUPPORTED
