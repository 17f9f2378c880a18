"""The forward kernels and MSS at benchmark scale against the float64 oracle.

The other forward tests use records of at most a few Mbp, on which a persistent CTA runs one or two units of
work.  The benchmark record (46.7 Mbp) gives every CTA of the two-tile kernel about 50 units, single-tile lead
units first, and its displaced last batch (prediction.py:105) lands in the middle of the record.  The full
float64 oracle is far too slow for such records, but a row's vote is the element-wise maximum over the windows
that cover it, so the oracle is exact on every row whose covering windows were all evaluated: `sampled_oracle`
runs it on a chosen set of windows and reports those complete rows.  The sets are blocks of windows around the
places where a kernel's schedule changes (CTA ranges, unit boundaries, the lead units, the displaced batch, the
record's end) and seeded random blocks."""
import ctypes

import numpy as np
import pytest

STEP, BATCH = 50, 256
CONFIG2_BASES = 46_700_000          # bench.py: the benchmark record
WT = 64                             # windows per tile of the tcgen05 kernels


# ------------------------------------------------------------------ the sampled oracle
def reference_windows(length, T, step, batch):
    """(start, placed row) of every window, restated from the reference: windows `range(0, L - T, step)`
    (deepgrp/prediction.py:31) in batches of `batch`, batch i voting at row i * len(batch) * step
    (prediction.py:105; a short last batch lands at its own length's multiple)."""
    starts = np.arange(0, max(length - T, 0), step, dtype=np.int64)
    place = np.empty(starts.size, dtype=np.int64)
    for i, b0 in enumerate(range(0, starts.size, batch)):
        nb = min(batch, starts.size - b0)
        place[b0:b0 + nb] = i * nb * step + np.arange(nb, dtype=np.int64) * step
    return starts, place


def coverage(place, T, rows):
    """Number of windows placed at `place` (rows place .. place + T - 1) that cover each of `rows`."""
    sp = np.sort(place)
    return np.searchsorted(sp, rows, "right") - np.searchsorted(sp, rows - T, "right")


def sampled_oracle(oracle, w, codes, step, batch, S, chunk=256):
    """The float64 oracle on the windows S only: (rows, votes float32[rows, C], complete bool[rows]).  `rows` are
    the rows S covers; a row is complete when every window that covers it is in S, so that its vote is the
    whole record's vote."""
    T, C = w.vecsize, w.n_classes
    starts, place = reference_windows(codes.size, T, step, batch)
    S = np.unique(np.asarray(S, dtype=np.int64))
    rows = np.unique((place[S][:, None] + np.arange(T)).ravel())
    votes = np.zeros((rows.size, C), dtype=np.float32)
    wd, eye = w.as_dict(), np.eye(5, dtype=np.float32)
    for k in range(0, S.size, chunk):
        ws = S[k:k + chunk]
        batch_x = eye[codes[starts[ws][:, None] + np.arange(T)]]
        probs = oracle.model_forward(batch_x, wd, dtype=np.float64).astype(np.float32)
        idx = np.searchsorted(rows, place[ws][:, None] + np.arange(T))
        np.maximum.at(votes, idx.ravel(), probs.reshape(-1, C))
    complete = coverage(place, T, rows) == coverage(place[S], T, rows)
    return rows, votes, complete


def onehot(codes):
    """int8[5, L] one-hot matrix of base codes 0..4 (A, C, G, T, N), as one_hot_encode_dna_sequence makes it."""
    fwd = np.zeros((5, codes.size), dtype=np.int8)
    fwd[codes, np.arange(codes.size)] = 1
    return fwd


@pytest.mark.parametrize("L,T,step,batch", [
    (3_000, 150, 50, 16),       # 57 windows: a short last batch of 9, displaced
    (2_000, 40, 60, 7),         # step > T: rows between windows are never covered
    (100, 150, 50, 16),         # L < T: no window at all
    (4_321, 37, 5, 64),         # dense overlap, 857 windows, last batch of 25
    (1_190, 150, 50, 4)])       # 21 windows, last batch of 1
def test_sampled_oracle_equals_full_oracle(oracle, L, T, step, batch):
    """With every window sampled the helper is the full float64 oracle, bit for bit; with a subset, its complete
    rows still are."""
    from deepgrp_b200 import model
    w = model.random_weights(T, 8, attention=True, seed=L).scaled(3.0)
    rng = np.random.default_rng(L)
    text = "".join(np.array(list("ACGTN"))[rng.integers(0, 5, size=L)])
    text = "A" + text[1:-1] + "C"
    _, fwd = oracle.one_hot_encode_dna_sequence(text)
    codes = fwd.argmax(axis=0).astype(np.uint8)
    exp = oracle.predict(lambda b: oracle.model_forward(b, w.as_dict(), dtype=np.float64).astype(np.float32),
                         oracle.fetch_validation_batch(fwd, step, batch, T), (L, 5), step)
    n = len(range(0, L - T, step))
    covered = np.flatnonzero((exp != 0).any(axis=1))
    rows, votes, complete = sampled_oracle(oracle, w, codes, step, batch, np.arange(n), chunk=16)
    assert complete.all() and np.array_equal(rows, covered)
    assert np.array_equal(votes.view(np.int32), exp[rows].view(np.int32))
    if n == 0:
        return
    S = np.concatenate([np.arange(0, min(n, 5)), np.arange(n // 2, min(n // 2 + 4, n)), np.arange(max(n - 3, 0), n)])
    rows, votes, complete = sampled_oracle(oracle, w, codes, step, batch, S, chunk=16)
    assert complete.any() and (step >= T or not complete.all())
    assert np.array_equal(votes[complete].view(np.int32), exp[rows[complete]].view(np.int32))


# ------------------------------------------------------------------ the kernels' schedules
def two_tile_schedule(n_windows, sm_count):
    """CTAs of gru_tc_attention_vote_kernel over one window range: grid (forward_tc.cu:464-467), contiguous tile
    range per CTA, `lead` single-tile units, then two-tile units, a single last tile (forward_tc.cu:156-169).
    -> [(tile_lo, tile_hi, lead, [(first tile, tiles) per unit])]"""
    n_tiles = -(-n_windows // WT)
    grid = min((n_tiles + 1) // 2, sm_count)
    ctas = []
    for b in range(grid):
        lo, hi = n_tiles * b // grid, n_tiles * (b + 1) // grid
        my = hi - lo
        lead = (b & 3) if my >= 32 else ((b & 1) if my >= 16 else 0)
        units, tile = [], lo
        while tile < hi:
            nt = 1 if (len(units) < lead or tile + 1 >= hi) else 2
            units.append((tile, nt))
            tile += nt
        ctas.append((lo, hi, lead, units))
    return ctas


def wide_schedule(n_windows, sm_count, ncta):
    """Groups (one CTA or a CTA pair) of rnn_tcw_kernel: grid (forward_tcw.cu:538-542), a contiguous unit range per
    group, unit u = tiles u * ncta + rank (forward_tcw.cu:218-222, 329-331).  -> (n_tiles, [(unit_lo, unit_hi)])"""
    n_tiles = -(-n_windows // WT)
    n_units = -(-n_tiles // ncta)
    groups = min(n_units, sm_count // ncta)
    return n_tiles, [(n_units * g // groups, n_units * (g + 1) // groups) for g in range(groups)]


def choose_windows(L, T, step, batch, required, optional, cap, seed, n_random=16):
    """Blocks of windows around the first windows of tiles: every `required` tile, the displaced last batch with the
    body windows under it, the record's last windows, `n_random` seeded random blocks, then a seeded subset of the
    `optional` tiles while the set stays below `cap` windows."""
    half = -(-T // step) + 1           # a block of 2 * half windows has complete rows on both sides of its centre
    _, place = reference_windows(L, T, step, batch)
    n = place.size
    full = n - n % batch
    S = set()

    def block(centre):
        return set(range(max(centre - half, 0), min(centre + half, n)))
    for tile in required:
        S |= block(tile * WT)
    if full < n:                       # the displaced batch and the body windows placed under its rows
        under = np.flatnonzero((place[:full] + T > place[full]) & (place[:full] < place[-1] + T))
        S |= set(range(full, n)) | set(range(max(under[0] - half, 0), min(under[-1] + 1 + half, full)))
    S |= set(range(max(full - 2 * half, 0), n))
    rng = np.random.default_rng(seed)
    for c in rng.integers(0, n, size=n_random):
        S |= block(int(c))
    assert len(S) <= cap, (len(S), cap)
    for tile in rng.permutation(np.array(sorted(set(optional) - set(required)), dtype=np.int64)):
        more = block(int(tile) * WT)
        if len(S | more) > cap:
            continue
        S |= more
    return np.array(sorted(S), dtype=np.int64)


def two_tile_boundaries(ctas):
    """(required, optional) tiles of the two-tile schedule: each CTA's first tile (its CTA boundary) is optional;
    for CTAs 0-3 and the last, every unit's first tile is optional, and the switch from the single-tile lead units
    to two-tile units and the last unit are required."""
    required, optional = set(), {lo for lo, _, _, _ in ctas}
    for b in sorted({0, 1, 2, 3, len(ctas) - 1} & set(range(len(ctas)))):
        lo, hi, lead, units = ctas[b]
        optional |= {t for t, _ in units}
        required |= {units[min(lead, len(units) - 1)][0], units[-1][0], min(hi, ctas[-1][1] - 1)}
    return sorted(required), sorted(optional)


# ------------------------------------------------------------------ forward cases
@pytest.fixture(scope="module")
def dg(gpu_ctx):
    import deepgrp_b200.model as model
    import deepgrp_b200.prediction as pred
    import deepgrp_b200.sharding as sharding

    class NS:
        pass
    ns = NS()
    ns.model, ns.pred, ns.sharding, ns.ctx = model, pred, sharding, gpu_ctx
    return ns


def windows_for_tiles(n_tiles, extra):
    """A window count with `n_tiles` tiles of 64, the last one holding `extra` windows (1..64)."""
    return (n_tiles - 1) * WT + extra


def length_for_windows(n, T, step=STEP, cut=0):
    """A record length with len(range(0, L - T, step)) == n (cut < step shortens it within that)."""
    L = T + n * step - cut
    assert len(range(0, L - T, step)) == n
    return L


def check_forward_at_scale(dg, oracle, name, w, codes, used_tc, tc_bound, S):
    """(a) the tcgen05 forward against the fp32 FFMA kernel on every row, (b) both against the sampled float64 oracle
    on its complete rows, (c) the never-covered rows, (d) argmax agreement.  Returns the measured maxima."""
    L, T, C = codes.size, w.vecsize, w.n_classes
    fwd = onehot(codes)
    ds = dg.pred.fetch_validation_batch(fwd, STEP, BATCH, T)
    tc = dg.pred.predict(w, ds, (L, C), STEP)
    assert dg.ctx.get_int("forward_used_tc") == used_tc
    dg.ctx.set_int("forward_tc", 0)
    try:
        f32 = dg.pred.predict(w, ds, (L, C), STEP)
        assert dg.ctx.get_int("forward_used_tc") == 0
    finally:
        dg.ctx.set_int("forward_tc", 1)
    del fwd, ds
    # (c) rows no window covers: zero in both, and exactly those (both placement families)
    _, place = reference_windows(L, T, STEP, BATCH)
    diff = np.zeros(L + T + 1, dtype=np.int32)
    np.add.at(diff, place, 1)
    np.add.at(diff, place + T, -1)
    never = np.cumsum(diff)[:L] == 0
    del diff, place
    assert np.array_equal((tc == 0).all(axis=1), never)
    assert np.array_equal((f32 == 0).all(axis=1), never)
    # (a), (d) every row
    d_tf = float(np.abs(tc - f32).max())
    agree_tf = float((tc.argmax(axis=1) == f32.argmax(axis=1)).mean())
    # (b) the sampled oracle
    rows, ref, complete = sampled_oracle(oracle, w, codes, STEP, BATCH, S)
    rc, ref = rows[complete], ref[complete]
    assert rc.size >= 1000
    d_tc = float(np.abs(tc[rc] - ref).max())
    d_f32 = float(np.abs(f32[rc] - ref).max())
    agree_tc = float((tc[rc].argmax(axis=1) == ref.argmax(axis=1)).mean())
    agree_f32 = float((f32[rc].argmax(axis=1) == ref.argmax(axis=1)).mean())
    print("%s: %d windows sampled, %d complete rows; max |dp| tcgen05 vs float64 %.3g, fp32 vs float64 %.3g, "
          "tcgen05 vs fp32 (all %d rows) %.3g; argmax agreement %.6f / %.6f / %.6f"
          % (name, len(S), rc.size, d_tc, d_f32, L, d_tf, agree_tc, agree_f32, agree_tf))
    assert d_tc < tc_bound
    assert d_f32 < 2e-5
    assert d_tf < tc_bound + 2e-5
    assert min(agree_tc, agree_f32, agree_tf) >= 0.9999
    return d_tc, d_f32, d_tf


def config2_codes():
    """The benchmark's record: bench.py synth_codes(46.7 M, [1, 0])."""
    return np.random.default_rng([1, 0]).integers(0, 4, size=CONFIG2_BASES, dtype=np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("scale,bound", [(1.0, 1e-6), (4.0, 1e-4)])
def test_config2_benchmark_record_vs_float64(dg, oracle, scale, bound):
    """The benchmark's inputs (T = 342, U = 60, random-init weights seed 0 and x4, the 46.7 Mbp record): about 99
    tiles and 50 units per CTA, the lead of b & 3 single-tile units, the displaced last batch mid-record."""
    T, U = 342, 60
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    if scale != 1.0:
        w = w.scaled(scale)
    codes = config2_codes()
    _, place = reference_windows(codes.size, T, STEP, BATCH)
    n = place.size
    ctas = two_tile_schedule(n, dg.ctx.get_int("sm_count"))
    assert min(hi - lo for lo, hi, _, _ in ctas) >= 32                      # lead = b & 3
    assert [c[2] for c in ctas[:4]] == [0, 1, 2, 3]
    assert len({hi - lo for lo, hi, _, _ in ctas}) == 2                     # CTA ranges of unequal length
    assert n % BATCH and T < place[-1] < codes.size // 2                    # the displaced batch lands mid-record
    required, optional = two_tile_boundaries(ctas)
    S = choose_windows(codes.size, T, STEP, BATCH, required, optional, cap=4096, seed=2)
    check_forward_at_scale(dg, oracle, "config 2, weights x%g" % scale, w, codes, 1, bound, S)


@pytest.mark.gpu
def test_two_tile_up32_lead_one_vs_float64(dg, oracle):
    """The <32> instantiation with 16-31 tiles per CTA (lead = b & 1) and CTA ranges of unequal length: an odd
    window, non-zero biases, ACGTN bases with N runs."""
    T, U = 151, 32
    sm = dg.ctx.get_int("sm_count")
    n_tiles = 23 * sm + sm // 2 + 1
    n = windows_for_tiles(n_tiles, 23)
    L = length_for_windows(n, T, cut=17)
    ctas = two_tile_schedule(n, sm)
    assert all(16 <= hi - lo < 32 for lo, hi, _, _ in ctas)                 # lead = b & 1
    assert len({hi - lo for lo, hi, _, _ in ctas}) == 2
    rng = np.random.default_rng(151)
    w0 = dg.model.random_weights(T, U, attention=True, seed=151)
    w = dg.model.ModelWeights(T, U, w0.kernel, w0.recurrent_kernel, rng.normal(0, 0.3, w0.bias.shape),
                              w0.ff_kernel, rng.normal(0, 0.3, w0.ff_bias.shape), w0.att_scale).scaled(2.0)
    codes = rng.integers(0, 5, size=L).astype(np.uint8)
    for a in rng.integers(100, L - 5000, size=300):                         # N runs of up to 4 kbp
        codes[a:a + int(rng.integers(1, 4000))] = 4
    codes[0], codes[-1] = 0, 1
    required, optional = two_tile_boundaries(ctas)
    S = choose_windows(L, T, STEP, BATCH, required, optional, cap=4096, seed=3)
    check_forward_at_scale(dg, oracle, "two-tile <32>, T 151", w, codes, 1, 2e-5, S)


def wide_boundaries(n_tiles, groups, ncta):
    """(required, optional) tiles of the wide schedule: every group's first tiles are optional; for groups 0-3 and
    the last, every unit's tiles are optional, and the tiles of the second unit and the last unit are required."""
    required, optional = set(), set()
    for g, (u0, u1) in enumerate(groups):
        optional |= {u0 * ncta + r for r in range(ncta)}
        if g in (0, 1, 2, 3, len(groups) - 1):
            optional |= {u * ncta + r for u in range(u0, u1) for r in range(ncta)}
            required |= {u * ncta + r for u in (u0 + 1, u1 - 1) for r in range(ncta)}
    return sorted(t for t in required if t < n_tiles), sorted(t for t in optional if t < n_tiles)


@pytest.mark.gpu
def test_wide_pair_config5b_many_units_vs_float64(dg, oracle):
    """Config 5b (T = 512, U = 128: rnn_tcw_kernel<128, 0, true>, a CTA pair per unit) with >= 8 units per pair,
    pairs of unequal unit counts, and an odd tile count: the last unit's second CTA runs a dead tile."""
    T, U = 512, 128
    sm = dg.ctx.get_int("sm_count")
    pairs = sm // 2
    n_units = 8 * pairs + pairs // 2 + 1
    n = windows_for_tiles(2 * n_units - 1, 41)
    L = length_for_windows(n, T, cut=29)
    n_tiles, groups = wide_schedule(n, sm, 2)
    assert n_tiles % 2 == 1 and len(groups) == pairs
    assert min(u1 - u0 for u0, u1 in groups) >= 8 and len({u1 - u0 for u0, u1 in groups}) == 2
    w = dg.model.random_weights(T, U, attention=True, seed=5).scaled(3.0)
    codes = np.random.default_rng(512).integers(0, 4, size=L, dtype=np.uint8)
    required, optional = wide_boundaries(n_tiles, groups, 2)
    S = choose_windows(L, T, STEP, BATCH, required, optional, cap=2048, seed=5)
    check_forward_at_scale(dg, oracle, "config 5b", w, codes, 3, 2e-5, S)


@pytest.mark.gpu
def test_wide_lstm_many_units_vs_float64(dg, oracle):
    """LSTM at 60 units (rnn_tcw_kernel<64, 1, false>, one CTA per unit) with >= 8 units per CTA."""
    T, U = 342, 60
    sm = dg.ctx.get_int("sm_count")
    n = windows_for_tiles(8 * sm + sm // 2 + 3, 7)
    L = length_for_windows(n, T, cut=3)
    n_tiles, groups = wide_schedule(n, sm, 1)
    assert len(groups) == sm and min(u1 - u0 for u0, u1 in groups) >= 8
    w = dg.model.random_weights(T, U, attention=True, seed=11, rnn="LSTM").scaled(2.0)
    codes = np.random.default_rng(60).integers(0, 4, size=L, dtype=np.uint8)
    required, optional = wide_boundaries(n_tiles, groups, 1)
    S = choose_windows(L, T, STEP, BATCH, required, optional, cap=2048, seed=6)
    check_forward_at_scale(dg, oracle, "LSTM, 60 units", w, codes, 2, 3e-5, S)


# ------------------------------------------------------------------ the benchmark's device route and MSS
@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 4.0])
def test_config2_device_route_and_mss_bit_exact(dg, oracle, scale):
    """The benchmark's call (dgrp_predict_codes_dev on device-resident codes, then _results): its labels are the
    oracle's MSS of the GPU's own probabilities and its rows the oracle's segments of those labels, bit for bit.
    The chunked MSS converges without the sequential completion; on the x4 weights it needs several rounds, so
    the float64 running sum rounds and the chain's prediction of chunk states is what decides the result.  The
    8-way position-sharded route then gives the same labels and rows."""
    import torch
    from deepgrp_b200 import _lib
    T, U = 342, 60
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    if scale != 1.0:
        w = w.scaled(scale)
    ctx, lib = dg.ctx, _lib.lib()
    codes = config2_codes()
    L = codes.size
    h = w.device_handle(ctx)
    d_codes = torch.from_numpy(codes).cuda()
    n_rows = ctypes.c_int64(0)
    _lib.check(lib.dgrp_predict_codes_dev(ctx.handle, h, ctypes.c_void_p(d_codes.data_ptr()), L, STEP, BATCH, 1, 50,
                                          50, _lib.COMPAT_REFERENCE, ctypes.byref(n_rows)))
    rounds = ctx.get_int("mss_rounds")
    labels = np.empty(L, dtype=np.uint8)
    rows = np.empty((n_rows.value, 3), dtype=np.int64)
    _lib.check(lib.dgrp_predict_codes_dev_results(ctx.handle, _lib.ptr(labels), L, _lib.ptr(rows), n_rows.value))
    del d_codes
    print("config 2, weights x%g: %d MSS rounds, %d rows" % (scale, rounds, n_rows.value))
    assert rounds > 0                  # converged without the sequential completion
    if scale == 4.0:
        assert rounds >= 3
    probs = dg.pred.predict(w, dg.pred.fetch_validation_batch(onehot(codes), STEP, BATCH, T), (L, 5), STEP)
    sc, cl = dg.pred.mss_scores(probs)
    del probs
    exp = oracle.find_mss_relabel(sc, cl, 5, 50, 50)
    del sc, cl
    assert np.array_equal(labels, exp)
    exp_rows = oracle.yield_segments_array(exp.astype(np.int64), 0)
    exp_rows = exp_rows[exp_rows[:, 2] > 0]
    assert np.array_equal(rows, exp_rows)
    del exp, exp_rows
    # position-sharded: eight ranges with halo recompute, one of them holding the displaced batch's rows (its
    # launch carries the batch as a second window range), then MSS and segments over the gathered record
    _, place = reference_windows(L, T, STEP, BATCH)
    tail_lo, tail_hi = place[place.size - place.size % BATCH], place[-1] + T
    ranges = dg.sharding.split_positions(L, 8)
    assert any(a <= tail_lo and tail_hi <= b for a, b in ranges)
    parts = [dg.sharding.predict_range(w, codes, L, a, b, STEP, BATCH) for a, b in ranges]
    lab = np.concatenate([p[0] for p in parts])
    scores = np.concatenate([p[1] for p in parts])
    del parts
    out, rows2 = dg.sharding.finish_record(lab, scores, 5, True, 50, 50, 0)
    assert np.array_equal(out, labels)
    assert np.array_equal(np.stack([rows2["start"], rows2["end"], rows2["label"]], axis=1), rows)
