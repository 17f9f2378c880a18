"""Position-range prediction against the float64 oracle, on every forward kernel and vote form.

Chunk sharding (bench.py's `strong` and `config5b` sections) splits one record into ranges of positions:
`dgrp_predict_range[_dev]` computes the labels and scores of `[p0, p1)` from the windows whose placed rows touch
the range (the halo), and `dgrp_finish_record[_dev]` runs MSS and segments over the gathered result.  That route
has code no whole-record call runs: the choice of each range's windows in both placement families and of the bases
it needs (api.cu core_predict_range), codes that start partway into the record (`codes_base`), votes into rows
relative to `pred_row0`, the displaced last batch (prediction.py:105) as a second window range of the same launch,
and the gather pass that clips each slab's rows to the range.  Every range here gets only its minimal code slice,
inside a device buffer whose other bytes are another record's valid codes, so a read outside the slice changes
values instead of passing unnoticed."""
import contextlib
import ctypes

import numpy as np
import pytest

from test_gpu_scale import (WT, coverage, dg, length_for_windows, onehot, reference_windows,  # noqa: F401
                            sampled_oracle, two_tile_schedule, wide_schedule, windows_for_tiles)

BATCH = 256
REFERENCE, FIXED = 0, 1                 # DGRP_COMPAT_REFERENCE / DGRP_COMPAT_FIXED
SMEM_LIMIT = 227 * 1024                 # dynamic shared memory of one block
MARGIN = 1 << 16                        # poison bytes on either side of a slice (> any tile's code span)


# ------------------------------------------------------------------ which windows a range recomputes
def placement(L, T, step, batch, compat):
    """(start, placed row) of every window and the number of windows in the body family (placed at w * step);
    the others form the displaced last batch.  The fixed placement is one batch of all windows."""
    n = len(range(0, max(L - T, 0), step))
    starts, place = reference_windows(L, T, step, batch if compat == REFERENCE else max(n, 1))
    full = n - n % batch if compat == REFERENCE else n
    return starts, place, full


def range_windows(L, T, step, batch, compat, p0, p1):
    """(a0, a1, t0, t1, need_lo, need_hi) of positions [p0, p1): the body windows [a0, a1) and the displaced
    batch's windows [t0, t1) whose placed rows [place, place + T) meet [p0, p1), and the bases [need_lo, need_hi)
    those windows read.  A family no window of which touches the range is empty (a0 == a1, t0 == t1), and a range
    without windows needs no bases (need_lo == need_hi == p0)."""
    starts, place, full = placement(L, T, step, batch, compat)
    fams = []
    for lo, hi in ((0, full), (full, place.size)):
        pf = place[lo:hi]                                   # ascending within a family
        a = lo + int(np.searchsorted(pf, p0 - T, "right"))  # first window with place + T > p0
        b = lo + int(np.searchsorted(pf, p1, "left"))       # past the last window with place < p1
        fams.append((a, max(a, b)) if p1 > p0 else (a, a))
    (a0, a1), (t0, t1) = fams
    used = [(x, y) for x, y in fams if y > x]
    if not used:
        return a0, a1, t0, t1, p0, p0
    return a0, a1, t0, t1, min(int(starts[x]) for x, _ in used), max(int(starts[y - 1]) + T for _, y in used)


def brute_range_windows(L, T, step, batch, compat, p0, p1):
    """The same by scanning every window: (body set, displaced set, need_lo, need_hi)."""
    starts, place, full = placement(L, T, step, batch, compat)
    hit = [w for w in range(place.size) if max(place[w], p0) < min(place[w] + T, p1)]
    body, tail = [w for w in hit if w < full], [w for w in hit if w >= full]
    if not hit:
        return body, tail, p0, p0
    return body, tail, min(int(starts[w]) for w in hit), max(int(starts[w]) + T for w in hit)


def test_range_windows_equals_brute_force_scan():
    """range_windows against a scan over every window: 1 890 seeded ranges over records of 1-5 000 bases, windows,
    steps, batches and both placements; ranges that are empty, one row long, at 0 and at L."""
    rng = np.random.default_rng(1245)
    n_cases = 0
    for T in (5, 37, 150):
        for step in (1, 7, 50, T, 2 * T + 3):
            for batch in (1, 7, 256):
                for compat in (REFERENCE, FIXED):
                    for k in range(3):
                        L = int(rng.integers(1, 5001 if k else 2 * T + 2))     # one record around the window
                        p0 = int(rng.integers(0, L + 1))
                        kinds = [(p0, p0), (p0, min(p0 + 1, L)), (0, int(rng.integers(0, L + 1))),
                                 (int(rng.integers(0, L + 1)), L), (min(p0, L - 1), L), (0, L)]
                        p1 = int(rng.integers(p0, L + 1))
                        kinds.append((p0, p1))
                        for a, b in kinds:
                            a0, a1, t0, t1, lo, hi = range_windows(L, T, step, batch, compat, a, b)
                            body, tail, blo, bhi = brute_range_windows(L, T, step, batch, compat, a, b)
                            assert list(range(a0, a1)) == body and list(range(t0, t1)) == tail, (L, T, step, a, b)
                            assert (lo, hi) == (blo, bhi), (L, T, step, batch, compat, a, b)
                            n_cases += 1
    assert n_cases == 1890


# ------------------------------------------------------------------ the kernels' shared-memory vote
def smem_vote_mode(kernel, UP, rnn, T, step, C=5):
    """The vote form launch_tc_t (forward_tc.cu:440-459) and launch_tcw_t (forward_tcw.cu:519-533) choose for a
    tile: 1 = in the idle A operand, 2 = a region of its own, 0 = window probabilities to HBM; None = the step or
    window has no tcgen05 form.  `kernel`: "two_tile", "wide" or "pair"."""
    KP = UP + 16
    A = 128 * KP * 2
    if kernel == "two_tile":
        B = (3 * UP + 16) * KP * 2
        a_room = 2 * 2 * A

        def smem(wpp, code_span):
            return 2 * B + 2 * 2 * A + 4 * (10 * (3 * UP + 4) + 2 * UP + wpp * T) + 4 * code_span + 128
    else:
        G, ncta = (4 if rnn else 3), (2 if kernel == "pair" else 1)
        B = (G * UP + 16) // ncta * KP * 2
        a_room = 2 * A

        def smem(wpp, code_span):
            return 2 * B + 2 * A + 4 * ((0 if rnn else 10 * (UP + 4)) + UP + wpp * T) + 2 * code_span + 128
    span = (WT - 1) * step + T
    if span > 16384:
        return None
    code_span = (span + 15) & ~15
    wpp = WT
    while wpp > 8 and smem(wpp, code_span) > SMEM_LIMIT:
        wpp >>= 1
    if smem(wpp, code_span) > SMEM_LIMIT:
        return None
    vote = span * C * 4
    if vote <= a_room:
        return 1
    return 2 if smem(wpp, code_span) + vote <= SMEM_LIMIT else 0


def vote_region_bytes(T, step, C=5):
    """The bytes of shared memory that vote mode 2 adds to a launch: the tile's span of rows (forward_tc.cu:453)."""
    return ((WT - 1) * step + T) * C * 4


def test_smem_vote_modes_of_the_range_cases():
    """The restated limits put the cases' steps where the GPU tests expect them: the default step in the A operand,
    case b's step 37 in a region of its own, and the larger steps of cases a and d (and case g's 97) to HBM.  Cases
    a and d reach no region of their own at any step: their A operand and operands leave too little room."""
    assert smem_vote_mode("two_tile", 64, 0, 342, 50) == 1
    assert smem_vote_mode("two_tile", 64, 0, 342, 59) == 1 and smem_vote_mode("two_tile", 64, 0, 342, 60) == 0
    assert smem_vote_mode("pair", 128, 0, 512, 50) == 1 and smem_vote_mode("pair", 128, 0, 512, 51) == 0
    assert smem_vote_mode("two_tile", 32, 0, 151, 37) == 2
    assert smem_vote_mode("two_tile", 32, 0, 40, 97) == 0
    assert all(smem_vote_mode("two_tile", 64, 0, 342, s) in (0, 1, None) for s in range(1, 300))
    assert all(smem_vote_mode("pair", 128, 0, 512, s) in (0, 1, None) for s in range(1, 300))


# ------------------------------------------------------------------ cases
# name: T, U, step, scale, options, expected forward_used_tc, kernel (for smem_vote_mode), probability bound of the
# matching tests/test_gpu_scale.py case (the fp32 bound where none matches)
CASES = {
    "a": dict(T=342, U=60, step=50, scale=1.0, opts={}, used=1, kernel="two_tile", bound=1e-6),
    "b": dict(T=151, U=32, step=37, scale=2.0, opts={}, used=1, kernel="two_tile", bound=2e-5),
    "c": dict(T=150, U=60, step=50, scale=2.0, opts={"forward_wide": 1}, used=2, kernel="wide", bound=2e-5),
    "d": dict(T=512, U=128, step=50, scale=3.0, opts={}, used=3, kernel="pair", bound=2e-5),
    "e": dict(T=90, U=60, step=50, scale=2.0, opts={}, used=2, kernel="wide", bound=3e-5, rnn="LSTM"),
    "f": dict(T=150, U=32, step=50, scale=2.0, opts={"forward_tc": 0}, used=0, kernel=None, bound=2e-5),
    "g": dict(T=40, U=20, step=97, scale=2.0, opts={}, used=1, kernel="two_tile", bound=2e-5),
    "u100": dict(T=200, U=100, step=50, scale=2.0, opts={}, used=3, kernel="pair", bound=2e-5),
}
N_WINDOWS = windows_for_tiles(60, 37)   # 3 813: >= 3 tiles per range at 17 ranges; a displaced batch of 229


@contextlib.contextmanager
def options(ctx, **kv):
    old = {k: ctx.get_int(k) for k in kv}
    try:
        for k, v in kv.items():
            ctx.set_int(k, v)
        yield
    finally:
        for k, v in old.items():
            ctx.set_int(k, v)


def make_case(dg, name, step=None, n_windows=N_WINDOWS):
    """(spec, weights, codes) of a case with `n_windows` windows; `step` overrides the case's step."""
    s = dict(CASES[name])
    if step is not None:
        s["step"] = step
    T, U, step = s["T"], s["U"], s["step"]
    seed = sum(map(ord, name)) + T
    rng = np.random.default_rng(seed)
    w = dg.model.random_weights(T, U, attention=True, seed=seed, rnn=s.get("rnn", "GRU"))
    if name == "b":            # non-zero biases
        w = dg.model.ModelWeights(T, U, w.kernel, w.recurrent_kernel, rng.normal(0, 0.3, w.bias.shape), w.ff_kernel,
                                  rng.normal(0, 0.3, w.ff_bias.shape), w.att_scale)
    if s["scale"] != 1.0:
        w = w.scaled(s["scale"])
    L = length_for_windows(n_windows, T, step, cut=step // 3)
    codes = rng.integers(0, 5 if name == "b" else 4, size=L).astype(np.uint8)
    if name == "b":            # N runs of up to 2 kbp
        for a in rng.integers(100, L - 3000, size=40):
            codes[a:a + int(rng.integers(1, 2000))] = 4
    codes[0], codes[-1] = 0, 1
    return s, w, codes


class Ranges:
    """dgrp_predict_range_dev on one record; each call gets its minimal code slice, placed at its record offset in a
    device buffer that otherwise holds another seeded record of valid codes 0-4."""

    def __init__(self, dg, w, codes, step, compat, seed):
        import torch
        from deepgrp_b200 import _lib
        self.torch, self._lib, self.lib, self.ctx = torch, _lib, _lib.lib(), dg.ctx
        self.h, self.T, self.L, self.step, self.compat = w.device_handle(dg.ctx), w.vecsize, codes.size, step, compat
        self.d_codes = torch.from_numpy(codes).cuda()
        poison = np.random.default_rng(seed).integers(0, 5, size=codes.size + 2 * MARGIN, dtype=np.uint8)
        self.d_poison = torch.from_numpy(poison).cuda()

    def need(self, p0, p1):
        return range_windows(self.L, self.T, self.step, BATCH, self.compat, p0, p1)

    def call(self, p0, p1, codes_base=None, codes_len=None, whole=False, step=None):
        """Labels and scores (device tensors) of [p0, p1).  `whole`: the whole record at codes_base 0, as bench.py
        passes it; otherwise the poisoned slice [codes_base, codes_base + codes_len), by default the minimal one."""
        torch = self.torch
        n = max(p1 - p0, 0)
        lab = torch.empty(max(n, 1), dtype=torch.uint8, device="cuda")
        sc = torch.empty(max(n, 1), dtype=torch.float32, device="cuda")
        if whole:
            buf, ptr, base, ln = None, self.d_codes.data_ptr(), 0, self.L
        else:
            if codes_base is None:
                _, _, _, _, codes_base, hi = self.need(p0, p1)
                codes_len = hi - codes_base
            buf = self.d_poison.clone()
            buf[MARGIN + codes_base:MARGIN + codes_base + codes_len] = self.d_codes[codes_base:codes_base + codes_len]
            ptr, base, ln = buf.data_ptr() + MARGIN + codes_base, codes_base, codes_len
        torch.cuda.synchronize()
        self._lib.check(self.lib.dgrp_predict_range_dev(
            self.ctx.handle, self.h, ctypes.c_void_p(ptr), int(base), int(ln), self.L, int(p0), int(p1),
            int(self.step if step is None else step), BATCH, self.compat, ctypes.c_void_p(lab.data_ptr()),
            ctypes.c_void_p(sc.data_ptr())))
        self.ctx.synchronize()
        del buf
        return lab[:n], sc[:n]

    def gathered(self, cuts, whole=False, check_windows=True):
        """The concatenated labels and scores of the ranges between consecutive cuts (host arrays)."""
        torch = self.torch
        labs, scs = [], []
        for p0, p1 in zip(cuts[:-1], cuts[1:]):
            lab, sc = self.call(p0, p1, whole=whole)
            if check_windows and p1 > p0:
                a0, a1, t0, t1, _, _ = self.need(p0, p1)
                assert self.ctx.timings()["windows"] == (a1 - a0) + (t1 - t0), (p0, p1)
            labs.append(lab)
            scs.append(sc)
        return torch.cat(labs).cpu().numpy(), torch.cat(scs).cpu().numpy()


def landmarks(L, T, step, compat):
    """Rows where the route changes: the displaced batch's first placed row (reference placement), the first placed
    row of a tile of the whole-record launch mid-record (its tiles count from window 0), and the first row after the
    last window's rows."""
    _, place, full = placement(L, T, step, BATCH, REFERENCE)
    tail_base = int(place[full])
    _, place_c, _ = placement(L, T, step, BATCH, compat)
    tile_row = int(place[WT * (place.size // WT // 2)])
    last_row = int(place_c.max()) + T
    return tail_base, tile_row, last_row


def range_tile_row(L, T, step, compat, p0, k=2):
    """The first placed row of tile k of a range call that starts at row p0.  The call forms its tiles from its own
    first body window a0, so its tile boundaries are not those of the whole-record launch."""
    a0 = range_windows(L, T, step, BATCH, compat, p0, L)[0]
    assert a0 + (k + 1) * WT <= placement(L, T, step, BATCH, compat)[2]       # a body tile, placed at w * step
    return (a0 + k * WT) * step


def partitions(L, T, step, compat, seed):
    """name -> cuts (ascending, 0 first, L last; a repeated cut is an empty range).  "tile_edge-1/+0/+1" end a range
    one row before, at and one row after the first placed row of that range's own third tile, so the call's last
    tile holds no window, none, or one."""
    tail_base, tile_row, last_row = landmarks(L, T, step, compat)
    assert last_row <= L - 2
    mid = (tile_row + tail_base) // 2
    hand = [0, 0, 1, tile_row - 1, tile_row, tile_row + 1, mid, mid, mid + step // 2, tail_base - 1, tail_base,
            tail_base + 1, last_row, last_row, L - 1, L, L]
    if step > T:              # a range that starts inside the gap between two windows' rows
        _, place_c, _ = placement(L, T, step, BATCH, compat)
        k = place_c.size // 3
        hand += [int(place_c[k]) + T + 5, int(place_c[k + 1]) + 2]
    rng = np.random.default_rng(seed)
    out = {"split%d" % k: [a for a, _ in split_positions(L, k)] + [L] for k in (2, 3, 8, 17)}
    out["random"] = sorted([0, L] + [int(x) for x in rng.integers(0, L + 1, size=11)])
    out["hand"] = sorted(hand)
    edge = range_tile_row(L, T, step, compat, mid)
    assert mid < edge - 1 and edge + 1 < tail_base
    for d in (-1, 0, 1):
        out["tile_edge%+d" % d] = [0, mid, edge + d, L]
    return out


def split_positions(L, k):
    from deepgrp_b200 import sharding
    return sharding.split_positions(L, k)


def whole_record(dg, w, codes, step, compat):
    """Labels and float32 scores of pred.predict's whole-record probabilities, by the GPU score transform."""
    T = w.vecsize
    probs = dg.pred.predict(w, dg.pred.fetch_validation_batch(onehot(codes), step, BATCH, T), (codes.size, 5), step,
                            compat="reference" if compat == REFERENCE else "fixed")
    sc, cl = dg.pred.mss_scores(probs)
    return cl.astype(np.uint8), sc.astype(np.float32)


def score_f32(votes):
    """The float32 score transform of vote.cu:53-66 (class, score) on votes float32[n, C]."""
    cls = votes.argmax(axis=1)
    m = np.minimum(votes.max(axis=1) + np.float32(1e-6), np.float32(0.99))
    t = np.log(m / (np.float32(1) - m))
    return cls, np.where(cls > 0, t, np.float32(-10) * t).astype(np.float32)


# The transform's slope: dt/dm = 1 / (m (1 - m)) on m = max(p) + 1e-6 in [1/C, 0.99], largest at 0.99 (101.01);
# class 0 scales the score by 10.  A row whose argmax agrees moves by at most that times the probability error.
SCORE_SLOPE = 10 / (0.99 * 0.01)
NEVER_SCORE = np.float32(-10) * np.log(np.float32(1e-6) / (np.float32(1) - np.float32(1e-6)))


def windows_near(place, T, rows, reach):
    """Windows whose placed rows meet [x - reach, x + reach) for any x in `rows`: every row within `reach` of x is
    then complete in sampled_oracle."""
    sp = np.argsort(place, kind="stable")
    ps = place[sp]
    S = [sp[np.searchsorted(ps, x - reach - T, "right"):np.searchsorted(ps, x + reach, "left")] for x in rows]
    return np.unique(np.concatenate(S))


def check_oracle(oracle, w, codes, step, compat, labels, scores, rows_of_interest, reach, bound, name,
                 min_rows_each=0):
    """Labels and scores on the complete rows of the sampled oracle around `rows_of_interest`: argmax agreement
    >= 99.99 %, and on agreeing rows the score within SCORE_SLOPE * bound (+ 4 float32 ulps of the transform) of
    the float32 transform of the oracle's votes.  Returns (largest |dscore|, agreement, complete rows)."""
    L, T = codes.size, w.vecsize
    _, place, _ = placement(L, T, step, BATCH, compat)
    S = windows_near(place, T, rows_of_interest, reach)
    batch = BATCH if compat == REFERENCE else max(place.size, 1)
    rows, votes, complete = sampled_oracle(oracle, w, codes, step, batch, S)
    rc, v = rows[complete], votes[complete]
    for x in rows_of_interest:
        assert np.count_nonzero(np.abs(rc - x) <= reach) >= min_rows_each, (name, x)
    ocls, osc = score_f32(v)
    agree = labels[rc] == ocls
    d = np.abs(scores[rc].astype(np.float64) - osc.astype(np.float64))[agree]
    tol = SCORE_SLOPE * bound + 4 * np.spacing(np.abs(osc[agree]))
    print("%s: %d windows, %d complete rows; max |dscore| %.3g (bound %.3g); argmax agreement %.6f"
          % (name, S.size, rc.size, d.max(initial=0.0), SCORE_SLOPE * bound, agree.mean()))
    assert rc.size >= 1000
    assert agree.mean() >= 0.9999
    assert (d <= tol).all(), (name, float(d.max()))
    return float(d.max(initial=0.0)), float(agree.mean()), rc


# ------------------------------------------------------------------ 2. ranges on every kernel
RANGE_CASES = [("a", REFERENCE), ("a", FIXED), ("b", REFERENCE), ("c", REFERENCE), ("d", REFERENCE),
               ("d", FIXED), ("e", REFERENCE), ("f", REFERENCE), ("f", FIXED), ("g", REFERENCE),
               ("u100", REFERENCE)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,compat", RANGE_CASES, ids=["%s-%s" % (n, "ref" if c == REFERENCE else "fixed")
                                                          for n, c in RANGE_CASES])
def test_ranges_equal_whole_record_and_oracle(dg, oracle, name, compat):
    """Every partition of the record into ranges, each range given only its poisoned minimal code slice, gives the
    whole record's labels and scores bit for bit; at every cut, the displaced batch and random rows they match the
    float64 oracle; never-covered rows score as an all-zero vote; short slices and bad ranges are refused."""
    from deepgrp_b200 import _lib, sharding
    s, w, codes = make_case(dg, name)
    T, step, L = s["T"], s["step"], codes.size
    with options(dg.ctx, **s["opts"]):
        exp_lab, exp_sc = whole_record(dg, w, codes, step, compat)
        assert dg.ctx.get_int("forward_used_tc") == s["used"]
        R = Ranges(dg, w, codes, step, compat, seed=L)
        parts = partitions(L, T, step, compat, seed=L)
        for pname, cuts in parts.items():
            lab, sc = R.gathered(cuts)
            assert dg.ctx.get_int("forward_used_tc") == s["used"], pname
            assert np.array_equal(lab, exp_lab), pname
            assert np.array_equal(sc.view(np.int32), exp_sc.view(np.int32)), pname
        # the host-pointer form on a few ranges, after a longer record left other codes in the context's buffer
        other = np.random.default_rng(L + 1).integers(0, 5, size=L + 10_000, dtype=np.uint8)
        sharding.predict_range(w, other, other.size, 0, 2 * T, step, BATCH, compat)
        tail_base, tile_row, last_row = landmarks(L, T, step, compat)
        for p0, p1 in [(0, 1), (tile_row - 1, tail_base + 1), (tail_base, last_row + 3), (L - 1, L)]:
            a0, a1, t0, t1, lo, hi = R.need(p0, p1)
            hl, hs = sharding.predict_range(w, codes[lo:hi], L, p0, p1, step, BATCH, compat, codes_base=lo)
            assert np.array_equal(hl, exp_lab[p0:p1]) and np.array_equal(hs.view(np.int32), exp_sc[p0:p1].view(np.int32))
        # refusals: a slice one base short at either end; a range past the record or reversed; step 0
        p0, p1 = next((a, b) for a, b in split_positions(L, 8) if a <= tail_base < b)
        a0, a1, t0, t1, lo, hi = R.need(p0, p1)
        assert a1 > a0 and (t1 > t0) == (compat == REFERENCE) and lo >= 1 and hi <= L - 1
        for base, ln in ((lo + 1, hi - lo - 1), (lo, hi - lo - 1)):
            with pytest.raises(_lib.DeepgrpError, match=r"needed bases \[%d, %d\)" % (lo, hi)):
                R.call(p0, p1, base, ln)
        for base, ln in ((lo - 1, hi - lo + 1), (lo, hi - lo + 1)):
            l2, s2 = R.call(p0, p1, base, ln)
            assert np.array_equal(l2.cpu().numpy(), exp_lab[p0:p1])
            assert np.array_equal(s2.cpu().numpy().view(np.int32), exp_sc[p0:p1].view(np.int32))
        for q0, q1, st in ((L - 5, L + 1, step), (10, 5, step), (0, 100, 0)):
            with pytest.raises(_lib.DeepgrpError):
                R.call(q0, q1, whole=True, step=st)
    # never-covered rows: class 0 and the score of an all-zero vote, bit for bit
    _, place, _ = placement(L, T, step, BATCH, compat)
    never = coverage(place, T, np.arange(L)) == 0
    assert never[last_row:].all()
    if name == "g":
        assert never[:last_row].any()                       # the gaps between windows
    assert (exp_lab[never] == 0).all() and (exp_sc[never].view(np.int32) == NEVER_SCORE.view(np.int32)).all()
    # the oracle around every cut, both edges of the displaced batch and seeded random rows
    cuts = sorted({c for cs in parts.values() for c in cs if 0 < c < last_row})
    _, place_r, full_r = placement(L, T, step, BATCH, REFERENCE)
    edges = [tail_base, int(place_r[-1]) + T]
    rnd = [int(x) for x in np.random.default_rng(L + 2).integers(T, last_row - T, size=4)]
    check_oracle(oracle, w, codes, step, compat, exp_lab, exp_sc, cuts + edges + rnd, 2 * step, s["bound"],
                 "case %s (%s)" % (name, "reference" if compat == REFERENCE else "fixed"))


# ------------------------------------------------------------------ 3. the vote forms of the range route
FORMS = [("default", {}), ("hbm", {"forward_smem_vote": 0}), ("hbm_slabs", {"forward_smem_vote": 0,
                                                                             "forward_slab_mb": 1}),
         ("atomic", {"forward_smem_vote": 0, "forward_gather": 0})]
FORM_WINDOWS = windows_for_tiles(8 * 4 * 4096 // WT, 37)   # > 3 slabs of 4 096 windows in each of 8 ranges
FORWARD_KERNELS = ("gru_tc_attention_vote_kernel", "rnn_tcw_kernel")


def forward_shared_memory(call):
    """The shared memory per block of the tcgen05 forward launches that `call` makes, as the CUDA profiler records
    it (static + dynamic bytes; the trace goes to a temporary directory)."""
    import json
    import os
    import tempfile
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    return {int(e["args"]["shared memory"]) for e in events
            if e.get("cat") == "kernel" and any(k in e.get("name", "") for k in FORWARD_KERNELS)}


FORM_CASES = [("a", None, 1), ("a", 60, 0), ("b", None, 2), ("d", None, 1), ("d", 51, 0), ("f", None, None)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,step,mode", FORM_CASES, ids=["%s-step%s" % (n, s or "default") for n, s, _ in FORM_CASES])
def test_range_vote_forms_agree_bit_for_bit(dg, name, step, mode):
    """The range route's vote forms give the same labels and scores as its default: window probabilities in HBM
    with the gather pass clipping each slab to the range and the displaced batch as a call of its own; the same in
    4 096-window slabs; the kernels' atomicMax straight into the range's rows.  The steps cover every shared-memory
    vote mode: in the A operand (1), a region of its own (2, case b) and none (0, by size)."""
    s, w, codes = make_case(dg, name, step, FORM_WINDOWS)
    T, step, L = s["T"], s["step"], codes.size
    # forward_slab_mb = 1 holds fewer than 4 096 windows of T x 5 float32, so slabs are 4 096 windows (forward.cu:350-351)
    assert T * 5 * 4 * 4096 > 1 << 20 and all(b - a > 3 * 4096 * step for a, b in split_positions(L, 8))
    if s["kernel"]:
        UP = 32 if s["U"] <= 32 else (64 if s["U"] <= 64 else 128)
        assert smem_vote_mode(s["kernel"], UP, 0, T, step) == mode
    R = Ranges(dg, w, codes, step, REFERENCE, seed=L + 3)
    tail_base, _, _ = landmarks(L, T, step, REFERENCE)
    parts = partitions(L, T, step, REFERENCE, seed=L)
    split8, hand = parts["split8"], parts["hand"]
    tail_range = next((a, b) for a, b in zip(split8[:-1], split8[1:]) if a <= tail_base < b)
    out = {}
    with options(dg.ctx, **s["opts"]):
        if mode is not None:
            # mode 2 launches with the vote region on top of the shared memory the HBM form launches with; modes 1 and
            # 0 launch with the same amount (the vote in the A operand, or no vote in shared memory)
            smem = {}
            for form, kv in FORMS[:2]:
                with options(dg.ctx, **kv):
                    smem[form] = forward_shared_memory(lambda: R.call(*tail_range))
            assert len(smem["default"]) == 1 and len(smem["hbm"]) == 1, smem
            extra = smem["default"].pop() - smem["hbm"].pop()
            assert extra == (vote_region_bytes(T, step) if mode == 2 else 0), (extra, mode)
        for form, kv in FORMS:
            with options(dg.ctx, **kv):
                out[form] = (R.gathered(split8), R.gathered(hand))
                assert dg.ctx.get_int("forward_used_tc") == s["used"], form
                R.call(*tail_range)
                launches = dg.ctx.timings()["kernel_launches"]
            if form == "default" and mode is not None:
                assert (launches == 2) == (mode != 0), launches   # one launch holds both families, then the score
            if form == "hbm":
                assert launches == (3 if s["used"] == 0 else 5), launches   # two forwards (+ two gathers), score
    ref = out["default"]
    for form, got in out.items():
        for (l0, s0), (l1, s1) in zip(ref, got):
            assert np.array_equal(l0, l1), form
            assert np.array_equal(s0.view(np.int32), s1.view(np.int32)), form


# ------------------------------------------------------------------ 4. the owner's finish
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "d"])
def test_finish_record_of_gathered_ranges_equals_oracle(dg, oracle, name):
    """dgrp_finish_record on the gathered labels and scores of 8 ranges: its labels are the oracle's MSS relabelling
    (or the labels themselves without MSS) and its rows the oracle's segments with label 0 removed, bit for bit, at
    several MSS settings and start positions.  dgrp_finish_record_dev is checked by its row count alone: it leaves
    its labels and rows on the device, and the C ABI has no call that returns them (dgrp_predict_codes_dev_results
    refuses them), so its labels are those of the host form, which runs the same code."""
    import torch
    from deepgrp_b200 import _lib, sharding
    s, w, codes = make_case(dg, name)
    T, step, L = s["T"], s["step"], codes.size
    R = Ranges(dg, w, codes, step, REFERENCE, seed=L + 4)
    lab, sc = R.gathered(parts8 := [a for a, _ in split_positions(L, 8)] + [L])
    assert len(parts8) == 9
    d_lab, d_sc = torch.from_numpy(lab).cuda(), torch.from_numpy(sc).cuda()
    for use_mss, mn, xd in ((1, 50, 50), (1, 1, 0), (1, 20, 5), (0, 50, 50)):
        exp = oracle.find_mss_relabel(sc.astype(np.float64), lab, 5, mn, xd) if use_mss else lab
        for startpos in (0, 17):
            out, rows = sharding.finish_record(lab, sc, 5, bool(use_mss), mn, xd, startpos)
            assert np.array_equal(out, exp), (use_mss, mn, xd)
            er = oracle.yield_segments_array(exp.astype(np.int64), startpos)
            er = er[er[:, 2] > 0]
            assert np.array_equal(np.stack([rows["start"], rows["end"], rows["label"]], axis=1), er)
        n_rows = ctypes.c_int64(0)
        torch.cuda.synchronize()
        _lib.check(_lib.lib().dgrp_finish_record_dev(dg.ctx.handle, ctypes.c_void_p(d_lab.data_ptr()),
                                                     ctypes.c_void_p(d_sc.data_ptr()), L, 5, use_mss, mn, xd,
                                                     ctypes.byref(n_rows)))
        assert n_rows.value == er.shape[0] > 0


# ------------------------------------------------------------------ 5. the benchmark's range sections at 248 Mbp
@pytest.mark.gpu
@pytest.mark.parametrize("section", ["strong", "config5b"])
def test_benchmark_range_sections_at_248mbp(dg, oracle, section):
    """bench.py's chunk-sharded sections on their exact inputs (synth_codes(248 M, [1, 0]), random-init weights seed
    0): 8 ranges on the whole device record (codes_base 0, as bench.py runs them) and on poisoned minimal slices
    equal one [0, L) range bit for bit; the finish equals dgrp_predict_codes_dev (dgrp_finish_record_dev by its row
    count, since the C ABI returns nothing else of it; the host form, which runs the same code, by labels and rows);
    around the 7 cuts, the displaced batch and the record's end the labels and scores match the float64 oracle."""
    import torch
    from deepgrp_b200 import _lib, sharding
    T, U, used, bound = (342, 60, 1, 1e-6) if section == "strong" else (512, 128, 3, 2e-5)
    step, L = 50, 248_000_000
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    codes = np.random.default_rng([1, 0]).integers(0, 4, size=L, dtype=np.uint8)     # bench.py synth_codes
    ctx, lib = dg.ctx, _lib.lib()
    sm = ctx.get_int("sm_count")
    ranges = split_positions(L, 8)
    cuts = [a for a, _ in ranges] + [L]
    R = Ranges(dg, w, codes, step, REFERENCE, seed=7)
    # each range's schedule: the two-tile kernel with >= 32 tiles per CTA (lead units b & 3), or >= 8 units per pair
    units = []
    for p0, p1 in ranges:
        a0, a1, t0, t1, _, _ = R.need(p0, p1)
        tiles = -(-(a1 - a0) // WT) + -(-(t1 - t0) // WT)
        if used == 1:
            ctas = two_tile_schedule(tiles * WT, sm)
            assert len(ctas) == sm and min(hi - lo for lo, hi, _, _ in ctas) >= 32
            units.append(max(len(u) for _, _, _, u in ctas))
        else:
            _, groups = wide_schedule(tiles * WT, sm, 2)
            assert len(groups) == sm // 2 and min(u1 - u0 for u0, u1 in groups) >= 8
            units.append(max(u1 - u0 for u0, u1 in groups))
    assert sum(t1 > t0 for p0, p1 in ranges for _, _, t0, t1, _, _ in [R.need(p0, p1)]) == 1
    print("%s: units per CTA/pair (largest) per range %s" % (section, units))
    res = {}
    for form in ("whole", "slice"):
        lab = torch.empty(L, dtype=torch.uint8, device="cuda")
        sc = torch.empty(L, dtype=torch.float32, device="cuda")
        for p0, p1 in ranges:
            l, s = R.call(p0, p1, whole=form == "whole")
            assert ctx.get_int("forward_used_tc") == used
            lab[p0:p1], sc[p0:p1] = l, s
            del l, s
        res[form] = (lab, sc)
    one = R.call(0, L, whole=True)
    for form in ("slice", "one"):
        l, s = one if form == "one" else res[form]
        assert torch.equal(l, res["whole"][0]) and torch.equal(s.view(torch.int32), res["whole"][1].view(torch.int32))
    del one, res["slice"]
    torch.cuda.synchronize()
    d_lab, d_sc = res["whole"]
    n_rows = ctypes.c_int64(0)
    _lib.check(lib.dgrp_finish_record_dev(ctx.handle, ctypes.c_void_p(d_lab.data_ptr()), ctypes.c_void_p(d_sc.data_ptr()),
                                          L, 5, 1, 50, 50, ctypes.byref(n_rows)))
    n_whole = ctypes.c_int64(0)
    _lib.check(lib.dgrp_predict_codes_dev(ctx.handle, R.h, ctypes.c_void_p(R.d_codes.data_ptr()), L, step, BATCH, 1,
                                          50, 50, REFERENCE, ctypes.byref(n_whole)))
    assert ctx.get_int("forward_used_tc") == used
    whole_lab = np.empty(L, dtype=np.uint8)
    whole_rows = np.empty((n_whole.value, 3), dtype=np.int64)
    _lib.check(lib.dgrp_predict_codes_dev_results(ctx.handle, _lib.ptr(whole_lab), L, _lib.ptr(whole_rows),
                                                  n_whole.value))
    assert n_rows.value == n_whole.value > 0
    lab, sc = d_lab.cpu().numpy(), d_sc.cpu().numpy()
    del d_lab, d_sc, res
    out, rows = sharding.finish_record(lab, sc, 5, True, 50, 50, 0)
    assert np.array_equal(out, whole_lab)
    assert np.array_equal(np.stack([rows["start"], rows["end"], rows["label"]], axis=1), whole_rows)
    del out, rows, whole_lab, whole_rows
    # the oracle: 1 200 rows around each cut, both edges of the displaced batch and the last covered rows
    _, place, full = placement(L, T, step, BATCH, REFERENCE)
    sites = cuts[1:-1] + [int(place[full]), int(place[-1]) + T, int(place[full - 1]) + T - 600]
    check_oracle(oracle, w, codes, step, REFERENCE, lab, sc, sites, 600, bound, section, min_rows_each=1000)
