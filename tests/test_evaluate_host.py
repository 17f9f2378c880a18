"""Evaluation against a repeat annotation without a GPU: the kernel logic of csrc/eval_core.cuh (the table
dgrp_evaluate_last builds and eval_confusion_kernel's windows, compiled for the host) against a numpy painter, the
annotation reader against preprocess_y, the metrics and the `deepgrp evaluate` command line."""
import argparse
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest

from deepgrp_b200 import __main__ as cli
from deepgrp_b200 import model as dgmodel
from deepgrp_b200 import prediction as dgpred
from deepgrp_b200 import preprocessing as dgprep

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BLOCK = 128 * 256


def paint_counts(C, span, rows, ann):
    """The independent painter: one label per position of the span [startpos, startpos + length) -- the row's label
    where a row covers it, the lowest class among the annotations that cover it for the truth -- then a bincount."""
    sp, length = span
    truth = np.zeros(length, np.int64)
    pred = np.zeros(length, np.int64)
    for b, e, c in sorted((tuple(int(v) for v in a) for a in ann), key=lambda t: -t[2]):
        truth[max(b - sp, 0):max(e - sp, 0)] = c
    for s, e, lab in rows:
        pred[s - sp:e - sp] = lab
    return np.bincount(truth * C + pred, minlength=C * C).reshape(C, C)


@pytest.fixture(scope="module")
def host_eval():
    so = os.path.join(HERE, "host", "libeval_host.so")
    src = os.path.join(HERE, "host", "eval_host.cpp")
    core = os.path.join(ROOT, "deepgrp_b200", "csrc", "eval_core.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(core)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    lib = ctypes.CDLL(so)
    lib.eval_host_counts.restype = ctypes.c_int64
    lib.eval_host_counts.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 6 + [ctypes.c_int64, ctypes.c_void_p]

    def counts(C, spans, rows, anns):
        """spans: [(startpos, length)]; rows / anns: per record, lists of (start, end, label) triples."""
        P = lambda a: ctypes.c_void_p(a.ctypes.data)            # noqa: E731
        tri = np.array([r for rr in rows for r in rr] or [(0, 0, 0)], np.int64).reshape(-1, 3)
        ann = np.array([a for aa in anns for a in aa] or [(0, 0, 0)], np.int64).reshape(-1, 3)
        row_off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
        ann_off = np.concatenate([[0], np.cumsum([len(a) for a in anns])]).astype(np.int64)
        sp = np.array([s for s, _ in spans] or [0], np.int64)
        ln = np.array([n for _, n in spans] or [0], np.int64)
        out = np.zeros((max(len(spans), 1), C, C), np.int64)
        blocks = lib.eval_host_counts(C, P(tri), P(row_off), P(ann), P(ann_off), P(sp), P(ln), len(spans), P(out))
        assert blocks == sum((n + BLOCK - 1) // BLOCK for _, n in spans)
        return out[:len(spans)]
    return counts


def random_rows(rng, C, sp, length, edges=False):
    """Disjoint, sorted rows inside the span, labels in [1, C); with `edges` the cuts sit on thread windows."""
    if length == 0:
        return []
    if edges:
        cuts = {sp + k * 128 + d for k in range(length // 128 + 1) for d in (-1, 0, 1)}
    else:
        cuts = set((sp + rng.integers(0, length + 1, size=int(rng.integers(0, 40)))).tolist())
    cuts = sorted({c for c in cuts if sp <= c <= sp + length} | {sp, sp + length})
    return [(a, b, int(rng.integers(1, C))) for a, b in zip(cuts, cuts[1:]) if a < b and rng.random() < 0.6]


def random_ann(rng, C, sp, length, n, spill=True):
    """Overlapping annotations of every class, some past both ends of the span, some empty (begin >= end)."""
    lo, hi = (max(0, sp - 300), sp + length + 300) if spill else (sp, sp + length)
    out = []
    for _ in range(n):
        b = int(rng.integers(lo, hi + 1))
        e = b + int(rng.integers(-3, 400))
        out.append((b, max(e, 0), int(rng.integers(1, C))))
    return out


@pytest.mark.parametrize("C", [2, 3, 4, 5])
def test_kernel_logic_equals_painter_random(host_eval, C):
    rng = np.random.default_rng(C)
    spans, rows, anns = [], [], []
    for length in [1, 127, 128, 129, BLOCK - 1, BLOCK, BLOCK + 1, 0, 5000, 2 * BLOCK + 77]:
        sp = int(rng.integers(0, 200))
        spans.append((sp, length))
        rows.append(random_rows(rng, C, sp, length))
        anns.append(random_ann(rng, C, sp, length, int(rng.integers(0, 200))))
    got = host_eval(C, spans, rows, anns)
    for r in range(len(spans)):
        want = paint_counts(C, spans[r], rows[r], anns[r])
        assert np.array_equal(got[r], want), (r, spans[r])
        assert got[r].sum() == spans[r][1]


@pytest.mark.parametrize("length", [1, 127, 128, 129, BLOCK - 1, BLOCK + 1])
def test_kernel_logic_window_edges(host_eval, length):
    """Rows and annotation runs that start or end at, one before and one after every thread window boundary, runs
    that touch (merged) and runs that cover the whole span and more."""
    rng = np.random.default_rng(length)
    C, sp = 5, 3
    rows = random_rows(rng, C, sp, length, edges=True)
    ann = [(a, b, int(rng.integers(1, C))) for a, b, _ in random_rows(rng, C, sp, length, edges=True)]
    ann += [(a, b, 2) for a, b, _ in rows[:20]] + [(0, sp + length + 10, 4), (sp + length, sp + length + 5, 1)]
    got = host_eval(C, [(sp, length)], [rows], [ann])
    assert np.array_equal(got[0], paint_counts(C, (sp, length), rows, ann))


def test_kernel_logic_several_records(host_eval):
    """Blocks never straddle records: many short and a few long records, the annotation of one record does not
    leak into the next."""
    rng = np.random.default_rng(7)
    C = 4
    spans = [(int(rng.integers(0, 50)), int(n)) for n in rng.choice([0, 1, 60, 128, 300, BLOCK + 3, 70000], 40)]
    rows = [random_rows(rng, C, sp, n) for sp, n in spans]
    anns = [random_ann(rng, C, sp, n, 50) for sp, n in spans]
    got = host_eval(C, spans, rows, anns)
    for r, (span, rr, aa) in enumerate(zip(spans, rows, anns)):
        assert np.array_equal(got[r], paint_counts(C, span, rr, aa)), r


# ---- the annotation reader --------------------------------------------------------------------------------
def test_read_annotation(tmp_path):
    path = tmp_path / "ann.txt"
    path.write_text("chr1 5 10 2 X 7 extra\n  chr2\t6 11 1\nchr1 13 15 4\nchr1 16 18 7 X\nchr1 20 20 1\n"
                    "chr1 30 25 2\n\nchr10 0 3 1 y\nchr1 1 4 1\n")
    got = dgprep.read_annotation(str(path), [1, 2, 4])
    assert list(got) == ["chr1", "chr2", "chr10"]
    assert all(a.dtype == np.int64 and a.shape[1] == 3 for a in got.values())
    assert got["chr1"].tolist() == [[5, 10, 2], [13, 15, 4], [20, 20, 1], [30, 25, 2], [1, 4, 1]]
    assert got["chr2"].tolist() == [[6, 11, 1]] and got["chr10"].tolist() == [[0, 3, 1]]
    assert dgprep.read_annotation(str(path), [3]) == {}
    for bad in ("chr1 -1 4 1\n", "chr1 1 -4 1\n", "chr1 1 x 1\n", "chr1 1.5 4 1\n", "chr1 1 4 one\n",
                "chr1 1 4 1\nchr2 1 4\n"):
        path.write_text(bad)
        with pytest.raises(ValueError):
            dgprep.read_annotation(str(path), [1])
    path.write_text("")
    assert dgprep.read_annotation(str(path), [1]) == {}


def test_read_annotation_truth_equals_preprocess_y(tmp_path):
    """The truth the kernel paints (lowest class first) from read_annotation equals preprocess_y(...).argmax(0)."""
    rng = np.random.default_rng(3)
    lines = []
    for _ in range(400):
        b = int(rng.integers(0, 3000))
        lines.append("%s %d %d %d x\n" % (rng.choice(["chrA", "chrB"]), b, b + int(rng.integers(-5, 300)),
                                           int(rng.integers(1, 7))))
    path = tmp_path / "ann.txt"
    path.write_text("".join(lines))
    repeats = [1, 2, 3, 4]
    for chrom in ("chrA", "chrB"):
        y = dgprep.preprocess_y(str(path), chrom, 2800, repeats)
        ann = dgprep.read_annotation(str(path), repeats)[chrom]
        truth = np.zeros(2800, np.int64)
        for b, e, c in sorted(ann.tolist(), key=lambda t: -t[2]):
            truth[b:e] = c
        assert np.array_equal(y.argmax(axis=0), truth)


# ---- metrics and JSON -------------------------------------------------------------------------------------
def test_confusion_metrics_and_json():
    cnf = np.array([[50, 3, 0], [4, 20, 0], [0, 0, 0]], np.int64)
    got = dgpred.confusion_metrics(cnf)
    with np.errstate(divide="ignore", invalid="ignore"):
        want = dgpred._calculate_metrics(cnf)
    want["TotalACC"] = 70 / 77
    assert set(got) == set(want) == {"TPR", "TNR", "PPV", "NPV", "FPR", "FNR", "FDR", "ACC", "F1", "MCC", "TotalACC"}
    for k in want:
        np.testing.assert_array_equal(got[k], want[k])
    doc = json.loads(json.dumps(dgpred.jsonable({"confusion": cnf, "metrics": got})))
    assert doc["confusion"] == cnf.tolist()
    assert doc["metrics"]["TPR"][2] is None and doc["metrics"]["PPV"][2] is None      # 0/0
    assert doc["metrics"]["TPR"][0] == pytest.approx(50 / 53)
    assert doc["metrics"]["TotalACC"] == pytest.approx(70 / 77)
    empty = json.loads(json.dumps(dgpred.jsonable(dgpred.confusion_metrics(np.zeros((2, 2), np.int64)))))
    assert empty["TotalACC"] is None and empty["MCC"] is None and empty["ACC"] == [None, None]


# ---- command line -----------------------------------------------------------------------------------------
def test_cli_parses_evaluate():
    p = cli.CommandLineParser().parse_args(["-s", "30", "-b", "64", "-l", "20", "-x", "-1", "-v", "evaluate",
                                            "m.hdf5", "ann.txt", "a.fa", "b.fa.gz", "--output", "o.json",
                                            "--no_use_mss", "--repeats", "2", "1"])
    a = p.args
    assert (a.command, a.model, a.annotation, a.FASTA, a.output) == ("evaluate", "m.hdf5", "ann.txt",
                                                                     ["a.fa", "b.fa.gz"], "o.json")
    assert (a.step_size, a.batch_size, a.min_mss_length, a.xdrop_length, a.no_use_mss, a.repeats) == \
        (30, 64, 20, -1, True, [2, 1])
    assert p.verbose == 1
    d = cli.CommandLineParser().parse_args(["evaluate", "m.hdf5", "ann.txt", "a.fa"]).args
    assert (d.output, d.no_use_mss, d.repeats) == ("-", False, None)
    # the README form is still prediction, and `evaluate` is not rewritten into it
    r = cli.CommandLineParser().parse_args(["-s", "30", "model.hdf5", "x.fa"]).args
    assert (r.command, r.model, r.FASTA) == ("predict", "model.hdf5", ["x.fa"])


@pytest.mark.parametrize("repeats", [["0"], ["3"], ["1", "5"], ["-1"]])
def test_cli_refuses_repeats_outside_the_classes(tmp_path, repeats):
    mpath = str(tmp_path / "m.npz")
    dgmodel.random_weights(50, 4, n_classes=3).save_npz(mpath)
    out = tmp_path / "o.json"
    with pytest.raises(SystemExit) as e:
        cli.CommandLineParser().parse_args(["evaluate", mpath, "ann.txt", "a.fa", "--output", str(out),
                                            "--repeats", *repeats]).run()
    assert e.value.code == 2 and not out.exists()
    assert dgpred.searched_repeats(None, 3) == [1, 2] and dgpred.searched_repeats([2, 1, 2], 3) == [1, 2]


def test_cli_document(monkeypatch, tmp_path):
    """The JSON document: options, records in file order with their file, the total the sum of the records; the
    annotation is read once with the searched numbers; nothing is written when a file fails."""
    mpath = str(tmp_path / "m.npz")
    dgmodel.random_weights(50, 4, n_classes=3).save_npz(mpath)
    ann = tmp_path / "ann.txt"
    ann.write_text("chr1 0 10 1\nchr1 5 8 2\n")
    files = {}
    for name, text in (("a.fa", b">chr1 x\nACGT\n>chr2\nAC\n"), ("b.fa", b">chr3\nGG\n")):
        files[name] = str(tmp_path / name)
        with open(files[name], "wb") as fh:
            fh.write(text)
    seen = []

    def fake(model, raw, annotation, step, batch, use_mss, min_len, xdrop, repeats):
        assert model.n_classes == 3 and (step, batch, use_mss, min_len, xdrop) == (50, 256, True, 50, 50)
        assert repeats == [1, 2] and annotation["chr1"].tolist() == [[0, 10, 1], [5, 8, 2]]
        k = len(seen)
        seen.append(bytes(raw))
        if b"fail" in bytes(raw):
            raise ValueError("negative dimensions are not allowed")
        recs = [{"header": "h%d%d" % (k, i), "chromosome": "c", "startpos": i, "length": 10,
                 "confusion": np.full((3, 3), k + i, np.int64), "metrics": dgpred.confusion_metrics(np.eye(3))}
                for i in range(2 - k)]
        tot = sum(r["confusion"] for r in recs)
        return {"classes": 3, "repeats": repeats, "records": recs,
                "total": {"confusion": tot, "metrics": dgpred.confusion_metrics(tot)}}
    monkeypatch.setattr(cli.dgpred, "evaluate_fasta", fake)
    out = tmp_path / "o.json"
    cli.CommandLineParser().parse_args(["evaluate", mpath, str(ann), files["a.fa"], files["b.fa"], "--output",
                                        str(out)]).run()
    doc = json.loads(out.read_text())
    assert (doc["classes"], doc["repeats"], doc["use_mss"], doc["step_size"]) == (3, [1, 2], True, 50)
    assert [(r["file"], r["header"]) for r in doc["records"]] == [(files["a.fa"], "h00"), (files["a.fa"], "h01"),
                                                                  (files["b.fa"], "h10")]
    assert doc["total"]["confusion"] == np.full((3, 3), 0 + 1 + 1).tolist()
    assert doc["total"]["metrics"]["TotalACC"] == pytest.approx(1 / 3)
    bad = tmp_path / "fail.fa"
    bad.write_bytes(b">fail\nNNN\n")
    out2 = tmp_path / "o2.json"
    with pytest.raises(ValueError):
        cli.CommandLineParser().parse_args(["evaluate", mpath, str(ann), files["a.fa"], str(bad), "--output",
                                            str(out2)]).run()
    assert not out2.exists()


def test_run_dispatches_evaluate(monkeypatch):
    parser = cli.CommandLineParser()
    parser.args = argparse.Namespace(command="evaluate", xdrop_length=7, batch_size=9, min_mss_length=11)
    seen = []
    monkeypatch.setattr(parser, "evaluate", lambda args, options: seen.append((args, options.batch_size)))
    parser.run()
    assert seen == [(parser.args, 9)]
