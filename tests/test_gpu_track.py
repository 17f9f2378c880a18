"""Probability tracks on the GPU (`keep_votes`, `dgrp_track_last`, `prediction.predict_fasta_tracks`,
`deepgrp predict --track`): byte for byte against the numpy restatement of the bedGraph contract applied to the GPU's
own votes (`prediction.predict` of each record), within rounding of the float64 oracle, and without side effects on
the TSV and the masked text."""
import io

import numpy as np
import pytest

from conftest import messy_fasta, random_dna, write_fasta
from test_track_host import restate_track

pytestmark = pytest.mark.gpu
BINS = (1, 10, 333)


@pytest.fixture(scope="module")
def dg(gpu_ctx):
    import deepgrp_b200.__main__ as cli
    import deepgrp_b200._lib as lib
    import deepgrp_b200.model as model
    import deepgrp_b200.prediction as pred
    import deepgrp_b200.sequence as seq

    class NS:
        pass
    ns = NS()
    ns.cli, ns.lib, ns.model, ns.pred, ns.seq, ns.ctx = cli, lib, model, pred, seq, gpu_ctx
    return ns


def record_votes(dg, model, raw, tmp_path, step=50, batch=256):
    """[(chromosome, startpos, votes float32[length, C])] of every record the reference reader yields (universal
    newlines, as `deepgrp predict --stepwise` opens the file), from prediction.predict of its one-hot matrix."""
    path = tmp_path / "votes.fa"
    path.write_bytes(raw)
    out = []
    with open(path, "r") as fh:
        for header, seq in dg.cli._read_multi_fasta(fh):
            startpos, fwd = dg.seq.one_hot_encode_dna_sequence(seq)
            n = fwd.shape[1]
            ds = dg.pred.fetch_validation_batch(fwd, step, batch, model.vecsize)
            out.append((header.split()[0], startpos, dg.pred.predict(model, ds, (n, model.n_classes), step)))
    return out


def sliced_tracks(dg, model, raw, bin):
    """{class: bytes} of predict_fasta_sliced with MSS on and a TSV stream, as the CLI runs --track."""
    streams = {c: io.BytesIO() for c in range(1, model.n_classes)}
    dg.pred.predict_fasta_sliced(model, raw, "f.fa", io.BytesIO(), 50, 256, True, 50, 50, trackstreams=streams,
                                 track_bin=bin)
    return {c: b.getvalue() for c, b in streams.items()}


def restated(records, C, bin):
    return {c: b"".join(restate_track(ch, sp, len(v), v[:, c], bin) for ch, sp, v in records) for c in range(1, C)}


def inputs():
    texts = [messy_fasta(seed).encode() for seed in range(5)]
    recs = [("edge N desc", "NNNN" + random_dna(3000, 1, "ACGTacgt") + "NNNNNNN"), ("", "ACGT" * 40),
            ("short", random_dna(100, 2)), ("  lead\tspace", "n" + random_dna(777, 3) + "N" * 50 + random_dna(90, 4)),
            ("tail", random_dna(2500, 5) + "NN")]
    texts.append("".join(">%s\n" % h + "\n".join(s[i:i + 61] for i in range(0, len(s), 61)) + "\n"
                         for h, s in recs).encode())
    return texts


ROUTES = {
    "two_tile_attention_c5": dict(T=150, U=32, attention=True, n_classes=5),
    "two_tile_no_attention_c5": dict(T=150, U=32, attention=False, n_classes=5),
    "two_tile_attention_c2": dict(T=150, U=32, attention=True, n_classes=2),
    "cta_pair_u100": dict(T=120, U=100, attention=True, n_classes=5),
    "lstm": dict(T=150, U=32, attention=True, n_classes=5, rnn="LSTM"),
    "fused_fallback": dict(T=150, U=32, attention=True, n_classes=5),
}


@pytest.mark.parametrize("route", sorted(ROUTES))
def test_tracks_equal_restatement_of_own_votes(dg, tmp_path, route):
    spec = dict(ROUTES[route])
    T, U = spec.pop("T"), spec.pop("U")
    model = dg.model.random_weights(T, U, seed=3, **spec).scaled(2.0 if spec.get("rnn") == "LSTM" else 4.0)
    C = model.n_classes
    smem = dg.ctx.get_int("forward_smem_vote")
    checked = 0
    try:
        if route == "fused_fallback":
            dg.ctx.set_int("forward_smem_vote", 0)      # vote + score fused: the route that never writes the votes
        for raw in inputs():
            try:
                records = record_votes(dg, model, raw, tmp_path)
            except IndexError:
                with pytest.raises(IndexError):
                    dg.pred.predict_fasta_tracks(model, raw, 50, 256, 10)
                continue
            for bin in BINS:
                got = dg.pred.predict_fasta_tracks(model, raw, 50, 256, bin)
                assert sorted(got) == list(range(1, C))
                want = restated(records, C, bin)
                for c in range(1, C):
                    assert got[c] == want[c], (route, bin, c)
            # with MSS, as `deepgrp predict --track` runs by default: the route that can fuse vote and score
            assert sliced_tracks(dg, model, raw, 10) == restated(records, C, 10), route
            checked += len(records)
        # one whole record with MSS: without keep_votes the fused fallback never writes the votes; with it, the
        # votes are materialised and the tracks still equal the restatement
        raw = (">f x\n" + random_dna(20000, 9) + "\n").encode()
        dg.pred._predict_fasta_call(model, raw, 50, 256, True, 50, 50, "reference")
        if route == "fused_fallback":
            assert dg.ctx.get_int("fused_last") == 1
        assert sliced_tracks(dg, model, raw, 10) == restated(record_votes(dg, model, raw, tmp_path), C, 10), route
        assert dg.ctx.get_int("fused_last") == 0
        if route == "cta_pair_u100":
            assert dg.ctx.get_int("forward_used_tc") == 3
    finally:
        dg.ctx.set_int("forward_smem_vote", smem)
    assert checked >= 8
    assert dg.ctx.get_int("keep_votes") == 0


def parse_bins(text, bin):
    """{chrom: (start positions of bins, values)} from bedGraph text, every line expanded into its bins."""
    out = {}
    for line in text.decode().splitlines():
        ch, s, e, v = line.split("\t")
        s, e = int(s), int(e)
        ks = np.arange(s // bin, (e - 1) // bin + 1)
        a, b = out.setdefault(ch, ([], []))
        a.append(ks)
        b.append(np.full(len(ks), float(v)))
    return {ch: (np.concatenate(a), np.concatenate(b)) for ch, (a, b) in out.items()}


@pytest.mark.parametrize("scale", (1.0, 4.0))
def test_tracks_against_float64_oracle(dg, oracle, scale):
    """defaults.toml shape (T = 342, U = 60, attention) on 1 Mbp with edge Ns: every bin value within the rounding
    (0.0005) plus 2e-5 of the oracle's binned votes."""
    T, U, L, bin = 342, 60, 1_000_000, 10
    w = dg.model.random_weights(T, U, attention=True, seed=0)
    if scale != 1.0:
        w = w.scaled(scale)
    seq = "N" * 13 + random_dna(L, 2) + "N" * 7
    raw = (">chrO x\n" + "\n".join(seq[i:i + 80] for i in range(0, len(seq), 80)) + "\n").encode()
    got = dg.pred.predict_fasta_tracks(w, raw, 50, 256, bin)
    startpos, fwd = dg.seq.one_hot_encode_dna_sequence(seq)
    wd = w.as_dict()
    exp = oracle.predict(lambda b: oracle.model_forward(b, wd, dtype=np.float64),
                         oracle.fetch_validation_batch(fwd, 50, 256, T), (L, 5), 50).astype(np.float64)
    k0 = startpos // bin
    nb = (startpos + L - 1) // bin - k0 + 1
    pad = np.full(nb * bin, np.nan)
    pad[startpos - k0 * bin:startpos - k0 * bin + L] = 0.0
    worst = 0.0
    for c in range(1, 5):
        pad[startpos - k0 * bin:startpos - k0 * bin + L] = exp[:, c]
        mean = np.nanmean(pad.reshape(nb, bin), axis=1)
        ks, vals = parse_bins(got[c], bin)["chrO"]
        assert np.array_equal(ks, np.arange(k0, k0 + nb))
        d = float(np.abs(vals - mean).max())
        worst = max(worst, d)
        assert d <= 0.0005 + 2e-5, (c, d)
    print("weights x%g: largest |track - oracle bin mean| %.3g" % (scale, worst))


# ------------------------------------------------------------------ side effects and the command line
@pytest.fixture(scope="module")
def model_path(dg, tmp_path_factory):
    p = str(tmp_path_factory.mktemp("m") / "w4.npz")
    dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0).save_npz(p)
    return p


def run_cli(dg, argv):
    dg.cli.CommandLineParser().parse_args(argv).run()


def read_tracks(prefix, C=5):
    return {c: open("%s.%d.bedGraph" % (prefix, c), "rb").read() for c in range(1, C)}


def test_no_side_effects(dg, tmp_path, model_path):
    a = tmp_path / "a.fa"
    a.write_bytes(inputs()[-1])
    b = tmp_path / "b.fa"
    write_fasta(str(b), [("chrB one", "NN" + random_dna(60000, 7)), ("chrC", random_dna(20000, 8, "ACGTacgtN"))])
    files = [str(a), str(b)]
    model = dg.model.load_model(model_path)
    want_tracks = {c: b"".join(dg.pred.predict_fasta_tracks(model, open(f, "rb").read(), 50, 256, 10)[c]
                               for f in files) for c in range(1, 5)}
    tracks = []
    for opts in ([], ["--no_use_mss"]):
        plain, masked = tmp_path / "plain.tsv", tmp_path / "plain.mask.fa"
        run_cli(dg, ["predict", model_path, *files, "--output", str(plain)] + opts)
        run_cli(dg, ["predict", model_path, *files, "--output", str(tmp_path / "m.tsv"), "--mask", str(masked)] + opts)
        run_cli(dg, ["predict", model_path, *files, "--output", str(tmp_path / "t.tsv"), "--track",
                     str(tmp_path / "t")] + opts)
        run_cli(dg, ["predict", model_path, *files, "--output", str(tmp_path / "tm.tsv"), "--track",
                     str(tmp_path / "tm"), "--mask", str(tmp_path / "tm.mask.fa")] + opts)
        ref = plain.read_bytes()
        assert ref.count(b"\n") > 10
        for name in ("m.tsv", "t.tsv", "tm.tsv"):
            assert (tmp_path / name).read_bytes() == ref, (opts, name)
        assert (tmp_path / "tm.mask.fa").read_bytes() == masked.read_bytes()
        tracks += [read_tracks(tmp_path / "t"), read_tracks(tmp_path / "tm")]
    for opts in (["-l", "7", "-x", "1"], ["-l", "500", "-x", "-1"]):
        run_cli(dg, opts + ["predict", model_path, *files, "--output", str(tmp_path / "o.tsv"), "--track",
                            str(tmp_path / "o")])
        tracks.append(read_tracks(tmp_path / "o"))
    for t in tracks:
        assert t == want_tracks
    run_cli(dg, ["predict", model_path, str(a), "--output", str(tmp_path / "b1.tsv"), "--track", str(tmp_path / "b1"),
                 "--track_bin", "1"])
    assert read_tracks(tmp_path / "b1") == dg.pred.predict_fasta_tracks(model, a.read_bytes(), 50, 256, 1)
    assert dg.ctx.get_int("keep_votes") == 0


def genome(rng, sizes):
    parts = []
    for i, n in enumerate(sizes):
        s = "N" * int(rng.integers(0, 40)) + random_dna(n, int(rng.integers(1 << 30)), "ACGTacgt")
        parts.append(">chr%d x\n" % i + "\n".join(s[j:j + 70] for j in range(0, len(s), 70)) + "\n")
    return parts


def test_multi_slice_file_equals_records_alone(dg):
    from deepgrp_b200.sharding import fasta_slices
    model = dg.model.random_weights(150, 32, attention=True, n_classes=4, seed=1).scaled(4.0)
    parts = genome(np.random.default_rng(4), [5_000_000, 1000, 4_000_000, 2500, 700])
    raw = "".join(parts).encode()
    assert len(raw) > 8 << 20 and len(fasta_slices(raw, 1)[0]) - 1 >= 2
    whole = dg.pred.predict_fasta_tracks(model, raw, 50, 256, 10)
    alone = [dg.pred.predict_fasta_tracks(model, p.encode(), 50, 256, 10) for p in parts]
    for c in range(1, 4):
        assert whole[c] == b"".join(a[c] for a in alone), c
        assert [line.split(b"\t")[0] for line in whole[c].splitlines()][-1] == b"chr4"


def test_error_in_later_slice_keeps_earlier_lines(dg, tmp_path, model_path):
    """A blank line in the second slice: IndexError, the TSV as the default route writes it, and the track files hold
    the lines of the first slice."""
    from deepgrp_b200.sharding import fasta_slices
    parts = genome(np.random.default_rng(6), [9_000_000, 3000, 2000])
    bad = "".join(parts[:2]) + parts[2].replace("\n", "\n\n", 3)
    raw = bad.encode()
    cuts = fasta_slices(raw, 1)[0]
    assert len(cuts) - 1 >= 2 and cuts[1] <= len(parts[0])
    path = tmp_path / "bad.fa"
    path.write_bytes(raw)
    with pytest.raises(IndexError):
        run_cli(dg, ["predict", model_path, str(path), "--output", str(tmp_path / "o.tsv"), "--track",
                     str(tmp_path / "t")])
    model = dg.model.load_model(model_path)
    first = dg.pred.predict_fasta_tracks(model, raw[:int(cuts[1])], 50, 256, 10)
    assert read_tracks(tmp_path / "t") == first and len(first[1]) > 0
    ref = io.BytesIO()
    with pytest.raises(IndexError):
        dg.pred.predict_fasta_tsv_stream(model, raw, str(path), ref, 50, 256, True, 50, 50)
    assert (tmp_path / "o.tsv").read_bytes() == ref.getvalue()
    with pytest.raises(ValueError):
        dg.pred.predict_fasta_tracks(model, b">a\nACGT\n>b\nNNNN\n", 50, 256, 10)


def test_refusals(dg):
    lib, ctx = dg.lib, dg.ctx
    model = dg.model.random_weights(150, 32, attention=True, n_classes=3, seed=0)
    raw = b">a x\nACGTACGTAC\n>\nAC\n>b\nGGGGACGTGGTT\n"

    def call(cls=1, bin=10, handle=None):
        text, n = lib.ctypes.c_void_p(), lib.ctypes.c_int64(0)
        rc = lib.lib().dgrp_track_last(handle or ctx.handle, cls, bin, lib.ctypes.byref(text), lib.ctypes.byref(n))
        return rc, lib.last_error()

    fresh = lib.Context(ctx.device)
    try:
        rc, err = call(handle=fresh.handle)
        assert rc == lib.E_ARG and "no dgrp_predict_fasta result to track" in err
    finally:
        fresh.close()
    dg.pred._predict_fasta_call(model, raw, 50, 256, True, 50, 50, "reference")
    rc, err = call()
    assert rc == lib.E_ARG and "did not keep its votes" in err
    ctx.set_int("keep_votes", 1)
    try:
        dg.pred._predict_fasta_call(model, raw, 50, 256, True, 50, 50, "reference")
        assert call()[0] == lib.OK and call(2, 1)[0] == lib.OK and call(1, 10**6)[0] == lib.OK
        for kwargs, msg in [(dict(cls=0), "class 0 is not in [1, 3)"), (dict(cls=3), "class 3 is not in [1, 3)"),
                            (dict(bin=0), "bin size 0"), (dict(bin=10**6 + 1), "bin size 1000001")]:
            rc, err = call(**kwargs)
            assert rc == lib.E_ARG and msg in err, (kwargs, err)
        # both records are shorter than a window: no vote, one line of zeros per record
        assert bytes(dg.pred.track_last(1, 4)) == b"a\t0\t10\t0.000\nb\t0\t12\t0.000\n"
        with pytest.raises(IndexError):
            dg.pred._predict_fasta_call(model, raw + b"\n\n>c\nACGT\n", 50, 256, True, 50, 50, "reference")
        rc, err = call()
        assert rc == lib.E_ARG and "no dgrp_predict_fasta result to track" in err          # a failed call
    finally:
        ctx.set_int("keep_votes", 0)
    with pytest.raises(ValueError):
        dg.pred.predict_fasta_tracks(model, raw, 50, 256, 0)
    # the slice loop restores the caller's keep_votes setting
    ctx.set_int("keep_votes", 1)
    try:
        dg.pred.predict_fasta_tracks(model, raw, 50, 256, 10)
        assert ctx.get_int("keep_votes") == 1
        dg.pred.predict_fasta_tsv_masked(model, raw, "f.fa", io.BytesIO(), io.BytesIO(), 50, 256, True, 50, 50)
        assert ctx.get_int("keep_votes") == 1 and call()[0] == lib.OK
    finally:
        ctx.set_int("keep_votes", 0)
    dg.pred.predict_fasta_tracks(model, raw, 50, 256, 10)
    assert ctx.get_int("keep_votes") == 0
    dg.pred._predict_fasta_call(model, raw, 50, 256, True, 50, 50, "reference")
    assert call()[0] == lib.E_ARG                                           # the votes were released


def test_scale_config2_record(dg):
    """One 20 Mbp record with the config-2 model shape, byte-exact against the restatement at bin 10."""
    C, L, T = 5, 20_000_000, 342
    model = dg.model.random_weights(T, 60, attention=True, seed=0)
    rng = np.random.default_rng(2)
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)]
    seq[:17] = ord("N")
    lines = np.concatenate([seq.reshape(-1, 100), np.full((L // 100, 1), ord("\n"), np.uint8)], axis=1)
    raw = b">chr21 synthetic\n" + lines.tobytes()
    got = dg.pred.predict_fasta_tracks(model, raw, 50, 256, 10)
    startpos, fwd = dg.seq.one_hot_encode_dna_sequence(seq.tobytes().decode())
    votes = dg.pred.predict(model, dg.pred.fetch_validation_batch(fwd, 50, 256, T), (fwd.shape[1], C), 50)
    for c in range(1, C):
        assert got[c] == restate_track("chr21", startpos, votes.shape[0], votes[:, c], 10), c
