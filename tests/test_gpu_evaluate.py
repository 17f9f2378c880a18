"""Evaluation against a repeat annotation on the GPU (`dgrp_evaluate_last`, `prediction.evaluate_fasta`,
`deepgrp evaluate`) against independent painters: one label per position from the prediction's rows and from the
annotation (lowest repeat number wins), then a bincount.  Every count comparison is exact."""
import gzip
import json

import numpy as np
import pytest

from conftest import messy_fasta, random_dna, write_fasta

pytestmark = pytest.mark.gpu
BLOCK = 128 * 256
LENGTHS = (1, 127, 128, 129, BLOCK - 1, BLOCK + 1)


@pytest.fixture(scope="module")
def dg(gpu_ctx):
    import deepgrp_b200._lib as lib
    import deepgrp_b200.model as model
    import deepgrp_b200.prediction as pred
    import deepgrp_b200.preprocessing as prep

    class NS:
        pass
    ns = NS()
    ns.lib, ns.model, ns.pred, ns.prep, ns.ctx = lib, model, pred, prep, gpu_ctx
    return ns


def weights(dg, C, T=150, U=32):
    return dg.model.random_weights(T, U, attention=True, n_classes=C, seed=0).scaled(4.0)


def cover(length, iv):
    """bool[length]: the union of the intervals iv (int64[n, 2], any order, clipped), without a per-interval loop."""
    d = np.zeros(length + 1, np.int64)
    iv = np.clip(np.asarray(iv, np.int64).reshape(-1, 2), 0, length)
    iv = iv[iv[:, 0] < iv[:, 1]]
    np.add.at(d, iv[:, 0], 1)
    np.add.at(d, iv[:, 1], -1)
    return np.cumsum(d[:-1]) > 0


def painter(C, startpos, length, rows, ann, repeats):
    """counts[t][p] of one record's span: rows = (start, end, label) triples, ann = (begin, end, number) triples, both
    in untrimmed coordinates."""
    rows = np.asarray(rows, np.int64).reshape(-1, 3)
    ann = np.asarray(ann, np.int64).reshape(-1, 3)
    pred = np.zeros(length, np.int64)
    for lab in range(1, C):
        pred[cover(length, rows[rows[:, 2] == lab, :2] - startpos)] = lab
    truth = np.zeros(length, np.int64)
    for c in sorted(repeats, reverse=True):
        truth[cover(length, ann[ann[:, 2] == c, :2] - startpos)] = c
    return np.bincount(truth * C + pred, minlength=C * C).reshape(C, C)


def expected(dg, C, model, raw, annotation, use_mss, repeats, opts=(50, 256, 50, 50)):
    step, batch, min_len, xdrop = opts
    rows, records = dg.pred.predict_fasta(model, raw, step, batch, use_mss, min_len, xdrop)
    out = []
    for r, (header, sp, ln) in enumerate(records):
        mine = rows[rows["record"] == r]
        tri = np.stack([mine["start"], mine["end"], mine["label"]], axis=1) if len(mine) else np.zeros((0, 3))
        out.append(painter(C, sp, ln, tri, annotation.get(header.split()[0], np.zeros((0, 3))), repeats))
    return out, records


def random_annotation(rng, names, length, n, numbers):
    """{chromosome: int64[n, 3]}: overlapping intervals of the given numbers, some past the record's ends or empty."""
    out = {}
    for name in names:
        b = rng.integers(0, length + 200, size=n)
        e = b + rng.integers(-5, 600, size=n)
        out[name] = np.stack([b, np.maximum(e, 0), rng.choice(numbers, size=n)], axis=1).astype(np.int64)
    return out


def evaluate(dg, model, raw, annotation, use_mss=True, repeats=None):
    return dg.pred.evaluate_fasta(model, raw, annotation, 50, 256, use_mss, 50, 50, repeats)


def messy_inputs():
    texts = [messy_fasta(seed).encode() for seed in range(8)]
    recs = [("len%d desc" % n, random_dna(n, n, "ACGTacgt")) for n in LENGTHS]
    recs.insert(2, ("", "ACGT" * 40))
    recs.insert(4, ("mid N", "NN" + random_dna(900, 1) + "N" * 300 + random_dna(700, 2) + "NNN"))
    parts = [">%s\r\n" % h + "\r\n".join(s[i:i + 61] for i in range(0, len(s), 61)) + "\r\n" for h, s in recs]
    texts.append("".join(parts).encode())
    return texts


@pytest.mark.parametrize("C,use_mss,repeats", [(2, True, None), (3, True, None), (3, False, None), (5, True, None),
                                               (5, False, None), (5, True, [1, 3])])
def test_counts_equal_painter(dg, C, use_mss, repeats):
    model = weights(dg, C)
    searched = list(range(1, C)) if repeats is None else repeats
    rng = np.random.default_rng(C * 10 + use_mss)
    checked = 0
    for raw in messy_inputs():
        names = {"chr%d" % i for i in range(4)} | {"x", "spaced", "h>h", "len1", "len127", "len128", "len129",
                                                   "len32767", "len32769", "mid"}
        annotation = random_annotation(rng, sorted(names), 40000, 120, np.arange(1, 6))
        try:
            want, records = expected(dg, C, model, raw, annotation, use_mss, searched)
        except IndexError:
            with pytest.raises(IndexError):
                evaluate(dg, model, raw, annotation, use_mss, repeats)
            continue
        got = evaluate(dg, model, raw, annotation, use_mss, repeats)
        assert got["classes"] == C and got["repeats"] == searched
        assert [(r["header"], r["startpos"], r["length"]) for r in got["records"]] == records
        for rec, w in zip(got["records"], want):
            assert rec["chromosome"] == rec["header"].split()[0]
            assert rec["confusion"].dtype == np.int64 and np.array_equal(rec["confusion"], w), rec["header"]
            assert rec["confusion"].sum() == rec["length"]
        assert np.array_equal(got["total"]["confusion"], sum(want) if want else np.zeros((C, C)))
        checked += len(records)
    assert checked >= 12


def test_reference_route(dg, tmp_path):
    """On a single-record file the total equals the reference's own evaluation: confusion_matrix of
    preprocess_y(...)[:, span].argmax(0) against the labels painted from the rows, and calculate_metrics."""
    C = 5
    model = weights(dg, C)
    seq = "NNNN" + random_dna(60000, 21, "ACGTacgt") + "NNNNNN"
    raw = (">chrQ some text\n" + "\n".join(seq[i:i + 60] for i in range(0, len(seq), 60)) + "\n").encode()
    rng = np.random.default_rng(5)
    lines = []
    for _ in range(300):
        b = int(rng.integers(0, 50000))
        lines.append("%s %d %d %d x\n" % (rng.choice(["chrQ", "chrZ"]), b, b + int(rng.integers(1, 900)),
                                           int(rng.integers(1, 7))))
    lines.append("chrQ 55000 55100 4\n")                                  # class 4 occurs in the truth
    path = tmp_path / "ann.txt"
    path.write_text("".join(lines))
    repeats = [1, 2, 3, 4]
    got = evaluate(dg, model, raw, dg.prep.read_annotation(str(path), repeats))
    rows, records = dg.pred.predict_fasta(model, raw, 50, 256, True, 50, 50)
    (_, sp, ln), = records
    truth = dg.prep.preprocess_y(str(path), "chrQ", len(seq), repeats)[:, sp:sp + ln].argmax(axis=0)
    pred = np.zeros(ln, np.int64)
    for s, e, lab in zip(rows["start"], rows["end"], rows["label"]):
        pred[s - sp:e - sp] = lab
    cnf, metrics = dg.pred.calculate_metrics(pred, truth)
    assert cnf.shape == (C, C)
    assert np.array_equal(got["total"]["confusion"], cnf)
    assert np.array_equal(got["records"][0]["confusion"], cnf)
    for k, v in metrics.items():
        np.testing.assert_array_equal(got["total"]["metrics"][k], v)


def test_oracle_rows(dg, oracle, tmp_path):
    """×4 weights of the config-1 shape: the oracle's TSV equals ours, and the counts from the oracle's rows equal the
    GPU's."""
    T, U, C = 150, 32, 5
    model = weights(dg, C, T, U)
    recs = [("chrA description", "NNN" + random_dna(30000, 1, "ACGTacgtn") + "NNNN"), ("chrB", random_dna(140, 2)),
            ("chrC", random_dna(12345, 3, "ACGTRYKM"))]
    path = tmp_path / "in.fa"
    write_fasta(str(path), recs)
    raw = path.read_bytes()
    ours = dg.pred.predict_fasta_tsv(model, raw, str(path), 50, 256, True, 50, 50)
    text = oracle.predict_fasta_tsv(str(path), model.as_dict(), T)
    assert text == ours and text.count("\n") > 20
    annotation = random_annotation(np.random.default_rng(9), ["chrA", "chrB", "chrC"], 31000, 300, np.arange(1, 5))
    got = evaluate(dg, model, raw, annotation)
    _, records = dg.pred.predict_fasta(model, raw, 50, 256, True, 50, 50)
    by_header = {}
    for line in text.splitlines():
        _, h, s, e, lab = line.split("\t")
        by_header.setdefault(h, []).append((int(s), int(e), int(lab)))
    for rec, (h, sp, ln) in zip(got["records"], records):
        want = painter(C, sp, ln, by_header.get(h, []), annotation[h.split()[0]], [1, 2, 3, 4])
        assert np.array_equal(rec["confusion"], want), h


def genome_text(rng, sizes):
    parts, names = [], []
    for i, n in enumerate(sizes):
        seq = np.frombuffer(random_dna(n, int(rng.integers(1 << 30)), "ACGTacgt").encode(), np.uint8).copy()
        seq[:int(rng.integers(0, 50))] = ord("N")
        names.append("chr%d" % i)
        s = seq.tobytes().decode()
        parts.append(">chr%d x\n" % i + "\n".join(s[j:j + 70] for j in range(0, len(s), 70)) + "\n")
    return parts, names


def test_slices_equal_records_alone(dg):
    from deepgrp_b200.sharding import fasta_slices
    C = 4
    model = weights(dg, C)
    rng = np.random.default_rng(14)
    parts, names = genome_text(rng, [5_000_000, 1000, 4_000_000, 2500, 3_000_000, 700])
    raw = "".join(parts).encode()
    assert len(raw) > 8 << 20 and len(fasta_slices(raw, 1)[0]) - 1 >= 2
    annotation = random_annotation(rng, names, 5_000_000, 20000, np.arange(1, C))
    whole = evaluate(dg, model, raw, annotation)
    assert [r["header"] for r in whole["records"]] == [n + " x" for n in names]
    for rec, part in zip(whole["records"], parts):
        alone = evaluate(dg, model, part.encode(), annotation)
        assert np.array_equal(rec["confusion"], alone["records"][0]["confusion"]), rec["header"]
    assert np.array_equal(whole["total"]["confusion"], sum(r["confusion"] for r in whole["records"]))


def test_scale_config2_record(dg):
    """A 46.7 Mbp record with the config-2 model shape and ~150 k overlapping annotations, exact against the
    vectorised painter."""
    C, L = 5, 46_700_000
    model = dg.model.random_weights(342, 60, attention=True, seed=0)
    rng = np.random.default_rng(2)
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)]
    lines = np.concatenate([seq.reshape(-1, 100), np.full((L // 100, 1), ord("\n"), np.uint8)], axis=1)
    raw = b">chr21 synthetic\n" + lines.tobytes()
    n = 150_000
    b = rng.integers(0, L, n)
    ann = np.stack([b, b + rng.integers(10, 6000, n), rng.integers(1, C, n)], axis=1).astype(np.int64)
    annotation = {"chr21": ann}
    got = evaluate(dg, model, raw, annotation)
    want, _ = expected(dg, C, model, raw, annotation, True, [1, 2, 3, 4])
    assert np.array_equal(got["records"][0]["confusion"], want[0])
    assert want[0][1:, 1:].sum() > 0


def test_refusals(dg):
    lib, ctx = dg.lib, dg.ctx
    model = weights(dg, 3)
    raw = b">a x\nACGTACGTAC\n>\nAC\n>b\nGGGGACGTGGTT\n"

    def call(C=3, ann=((0, 5, 1), (2, 7, 2)), off=(0, 2, 2), n=2):
        a = np.array(ann, np.int64).reshape(-1, 3)
        o = np.array(off, np.int64)
        out = np.zeros((max(n, 1), C, C), np.int64)
        rc = lib.lib().dgrp_evaluate_last(ctx.handle, C, lib.ptr(a), lib.ptr(o), n, lib.ptr(out))
        return rc, out, lib.last_error()

    fresh = lib.Context(ctx.device)
    try:
        a, o, out = np.zeros((1, 3), np.int64), np.zeros(3, np.int64), np.zeros((2, 3, 3), np.int64)
        assert lib.lib().dgrp_evaluate_last(fresh.handle, 3, lib.ptr(a), lib.ptr(o), 2, lib.ptr(out)) == lib.E_ARG
        assert "no dgrp_predict_fasta result to evaluate" in lib.last_error()
    finally:
        fresh.close()
    dg.pred.predict_fasta(model, raw, 50, 256, True, 50, 50)
    rc, out, _ = call()
    assert rc == lib.OK and out[0].sum() == 10 and out[1].sum() == 12 and out[1, 0].sum() == 12
    assert call()[0] == lib.OK                                              # may run again
    for kwargs, msg in [(dict(n=3, off=(0, 2, 2, 2)), "kept 2 records"), (dict(C=4), "model of 3 classes"),
                        (dict(ann=((0, 5, 3),)), "class 3 is not in [1, 3)"),
                        (dict(ann=((0, 5, 0),)), "class 0 is not in [1, 3)"),
                        (dict(ann=((-1, 5, 1),)), "negative coordinate"),
                        (dict(ann=((1, -5, 1),)), "negative coordinate"), (dict(off=(0, 2, 1)), "ann_off decreases")]:
        if "ann" in kwargs and "off" not in kwargs:
            kwargs["off"] = (0, 1, 1)
        rc, _, err = call(**kwargs)
        assert rc == lib.E_ARG and msg in err, (kwargs, err)
    a, o, out = np.zeros((1, 3), np.int64), np.zeros(3, np.int64), np.zeros((2, 3, 3), np.int64)
    for ptrs in [(None, lib.ptr(o), lib.ptr(out)), (lib.ptr(a), None, lib.ptr(out)), (lib.ptr(a), lib.ptr(o), None)]:
        assert lib.lib().dgrp_evaluate_last(ctx.handle, 3, *ptrs[:2], 2, ptrs[2]) == lib.E_ARG
        assert "must not be NULL" in lib.last_error()
    dg.pred.predict_fasta_tsv_sharded(model, raw, "f.fa", 50, 256, True, 50, 50, 0, 2)
    assert call()[0] == lib.E_ARG                                           # after a sharded call
    dg.pred.predict_fasta(model, raw, 50, 256, True, 50, 50)
    assert call()[0] == lib.OK
    dg.pred.mask_fasta(raw, np.zeros(0, lib.ROW_DTYPE))
    rc, _, err = call()
    assert rc == lib.E_ARG and "another call has used its buffers" in err   # the buffers were reused
    with pytest.raises(IndexError):
        dg.pred.predict_fasta(model, raw + b"\n\n>c\nACGT\n", 50, 256, True, 50, 50)
    assert call()[0] == lib.E_ARG                                           # a failed call


# ------------------------------------------------------------------ end to end through the CLI
@pytest.fixture(scope="module")
def model_path(dg, tmp_path_factory):
    p = str(tmp_path_factory.mktemp("m") / "w4.npz")
    weights(dg, 5).save_npz(p)
    return p


def run_cli(argv):
    from deepgrp_b200.__main__ import CommandLineParser
    CommandLineParser().parse_args(argv).run()


def test_cli_end_to_end(dg, tmp_path, model_path):
    rng = np.random.default_rng(31)
    parts, names = genome_text(rng, [70000, 3000, 45000])
    a = tmp_path / "a.fa"
    a.write_text("".join(parts[:2]))
    b = tmp_path / "b.fa.gz"
    with gzip.open(b, "wt") as fh:
        fh.write(parts[2].replace("chr2", "chr7"))
    ann = tmp_path / "ann.txt"
    lines = ["%s %d %d %d RM\n" % (c, s, s + int(rng.integers(5, 800)), int(rng.integers(1, 6)))
             for c in ("chr0", "chr1", "chr7", "chrX") for s in rng.integers(0, 70000, 300)]
    ann.write_text("".join(lines))
    out = tmp_path / "o.json"
    run_cli(["-v", "evaluate", model_path, str(ann), str(a), str(b), "--output", str(out), "--repeats", "1", "2", "4"])
    doc = json.loads(out.read_text())
    assert (doc["classes"], doc["repeats"], doc["use_mss"]) == (5, [1, 2, 4], True)
    assert [(r["file"], r["chromosome"]) for r in doc["records"]] == [(str(a), "chr0"), (str(a), "chr1"),
                                                                       (str(b), "chr7")]
    total = np.sum([r["confusion"] for r in doc["records"]], axis=0)
    assert doc["total"]["confusion"] == total.tolist() and total.sum() == sum(r["length"] for r in doc["records"])
    model = dg.model.load_model(model_path)
    annotation = dg.prep.read_annotation(str(ann), [1, 2, 4])
    want = dg.pred.evaluate_fasta(model, a.read_bytes(), annotation, 50, 256, True, 50, 50, [1, 2, 4])
    assert doc["records"][0]["confusion"] == want["records"][0]["confusion"].tolist()
    assert doc["records"][0]["metrics"] == json.loads(json.dumps(dg.pred.jsonable(want["records"][0]["metrics"])))


@pytest.mark.parametrize("kind,error", [("blank", IndexError), ("alln", ValueError)])
def test_cli_errors_write_nothing(dg, tmp_path, model_path, kind, error):
    good = tmp_path / "good.fa"
    good.write_text(">chr1\n" + random_dna(5000, 1) + "\n")
    bad = tmp_path / "bad.fa"
    bad.write_text(">chr1\nACGT\n\nACGT\n" if kind == "blank" else ">chr1\nACGTACGT\n>chr2\nNNNNNN\n")
    ann = tmp_path / "ann.txt"
    ann.write_text("chr1 0 100 1\n")
    out = tmp_path / "o.json"
    with pytest.raises(error):
        run_cli(["evaluate", model_path, str(ann), str(good), str(bad), "--output", str(out)])
    assert not out.exists()
