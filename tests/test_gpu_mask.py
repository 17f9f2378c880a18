"""Repeat-masked FASTA on the GPU (`dgrp_mask_fasta`, `dgrp_mask_fasta_last`, `deepgrp predict --mask`) against the
host restatement of the semantics in test_mask_host.py.  Every comparison is bit-exact."""
import random

import numpy as np
import pytest

from conftest import random_dna
from test_mask_host import all_texts, mask_fasta as oracle_mask, positions

pytestmark = pytest.mark.gpu
MODES = ("soft", "hard")


@pytest.fixture(scope="module")
def dg(gpu_ctx):
    import deepgrp_b200._lib as lib
    import deepgrp_b200.model as model
    import deepgrp_b200.prediction as pred

    class NS:
        pass
    ns = NS()
    ns.lib, ns.model, ns.pred, ns.ctx = lib, model, pred, gpu_ctx
    return ns


def random_rows(text: bytes, seed: int):
    """Seeded disjoint rows on every kept record: the first and the last position are covered, and some rows are
    adjacent.  -> (structured rows, {record: [(start, end)]})."""
    rng = random.Random(seed)
    rows, by_rec = [], {}
    for r, offs in enumerate(positions(text)):
        n = len(offs)
        if n == 0:
            continue
        cuts = sorted(set(rng.sample(range(1, n), min(n - 1, rng.randint(1, 12)))) | {0, n}) if n > 1 else [0, 1]
        pairs = list(zip(cuts, cuts[1:]))
        keep = [p for i, p in enumerate(pairs) if i in (0, len(pairs) - 1) or rng.random() < 0.6]
        by_rec[r] = keep
        rows += [(a, b, rng.randint(1, 4), r) for a, b in keep]
    import deepgrp_b200._lib as lib
    return np.array(rows, dtype=lib.ROW_DTYPE), by_rec


def lines(seq: str, widths, nl="\n"):
    out, i, k = [], 0, 0
    while i < len(seq):
        w = widths[k % len(widths)]
        out.append(seq[i:i + w])
        i += w
        k += 1
    return nl.join(out) + nl


def edge_texts():
    """Records and lines across the 4 096-byte tile and the 16-byte vector boundaries, 1-byte lines, lines longer
    than a tile, a file of headers only, and a multi-MB file."""
    out = []
    for pad in (1, 2, 15, 16, 17, 4095, 4096, 4097):
        out.append((">p\n" + "A" * pad + "\n>r\n" + lines(random_dna(9000, pad), [4093, 1, 17, 16])).encode())
    out.append((">one\n" + lines(random_dna(300, 1), [1]) + ">two\r\n" + lines(random_dna(200, 2), [1], "\r\n")).encode())
    out.append((">long\n" + lines(random_dna(3 * 4096 + 5, 3), [10000]) + ">x\n" + "acgtN" * 900 + "\n").encode())
    out.append(b"".join(b">h%d\n" % i for i in range(3000)))
    rng = np.random.default_rng(4)
    parts = ["pre amble\n"]
    for i in range(40):
        seq = random_dna(int(rng.integers(1, 200000)), 100 + i, "ACGTNacgt")
        parts.append(">" + ("rec%d" % i if i % 9 else "") + "\n" + lines(seq, [60, 61, 59]))
    out.append("".join(parts).encode())
    return out


def gpu(dg, text, rows, mode):
    return dg.pred.mask_fasta(text, rows, mode)


@pytest.mark.parametrize("mode", MODES)
def test_mask_fasta_matches_oracle(dg, mode):
    for i, text in enumerate(all_texts() + edge_texts()):
        rows, by_rec = random_rows(text, i)
        assert gpu(dg, text, rows, mode) == oracle_mask(text, by_rec, mode), i
        assert gpu(dg, text, rows[:0], mode) == text


def test_mask_fasta_unaligned_host_buffers(dg):
    text = edge_texts()[3]
    rows, by_rec = random_rows(text, 5)
    want = oracle_mask(text, by_rec, "soft")
    store = np.zeros(len(text) + 64, np.uint8)
    base = (-store.ctypes.data) % 16
    for off in range(1, 16):
        view = store[base + off:base + off + len(text)]
        view[:] = np.frombuffer(text, np.uint8)
        assert view.ctypes.data % 16 == off
        assert gpu(dg, view, rows, "soft") == want


def test_mask_fasta_refusals(dg):
    lib = dg.lib
    text = b">a\nACGTACGT\n>\nAC\n>b\nGGGG\n"
    R = lambda *t: np.array(list(t), dtype=lib.ROW_DTYPE)        # noqa: E731
    assert gpu(dg, text, R((0, 8, 1, 0), (0, 4, 2, 1)), "hard") == b">a\nNNNNNNNN\n>\nAC\n>b\nNNNN\n"
    bad = [R((0, 2, 1, 0), (1, 3, 1, 0)),            # overlap
           R((4, 6, 1, 0), (0, 2, 1, 0)),            # unsorted within a record
           R((0, 2, 1, 1), (0, 2, 1, 0)),            # unsorted records
           R((0, 9, 1, 0)),                          # past its record
           R((0, 5, 1, 1)),                          # past its record (the dropped record is not counted)
           R((0, 2, 1, 2)), R((0, 2, 1, -1)),        # record index
           R((0, 2, 0, 0)), R((-1, 2, 1, 0)), R((3, 3, 1, 0))]
    for rows in bad:
        with pytest.raises(lib.DeepgrpError) as e:
            gpu(dg, text, rows, "soft")
        assert e.value.code == lib.E_ARG
    with pytest.raises(ValueError):
        gpu(dg, text, R(), "upper")
    out = np.zeros(len(text), np.uint8)
    buf = np.frombuffer(text, np.uint8)
    assert lib.lib().dgrp_mask_fasta(dg.ctx.handle, lib.ptr(buf), len(text), None, 0, 2, lib.ptr(out)) == lib.E_ARG
    with pytest.raises(IndexError):
        gpu(dg, b">a\nAC\n\nGT\n", R(), "soft")


def mask_last(dg, raw, mode, n=None):
    lib = dg.lib
    buf = np.frombuffer(raw, np.uint8)
    out = np.zeros(max(len(raw), 1), np.uint8)
    rc = lib.lib().dgrp_mask_fasta_last(dg.ctx.handle, lib.ptr(buf), len(raw) if n is None else n,
                                        lib.MASK_HARD if mode == "hard" else lib.MASK_SOFT, lib.ptr(out))
    return rc, out[:len(raw)].tobytes()


def test_mask_fasta_last_equals_mask_fasta(dg):
    lib = dg.lib
    w = dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0)
    texts = [edge_texts()[-1], b"pre\r\n>a x\r\n" + lines(random_dna(30000, 9, "ACGTacgtN"), [70], "\r\n").encode()
             + b">\nACGT\n>b\nNNNN" + random_dna(5000, 10).encode() + b"NN"]
    for raw in texts:
        rows, _ = dg.pred.predict_fasta(w, raw, 50, 256, True, 50, 50)
        assert len(rows) > 20
        by_rec = {}
        for r in rows:
            by_rec.setdefault(int(r["record"]), []).append((int(r["start"]), int(r["end"])))
        for route in ("rows", "tsv"):
            for mode in MODES:
                if route == "rows":
                    dg.pred.predict_fasta(w, raw, 50, 256, True, 50, 50)
                else:
                    dg.pred.predict_fasta_tsv_view(w, raw, "f.fa", 50, 256, True, 50, 50)
                rc, got = mask_last(dg, raw, mode)
                assert rc == lib.OK
                assert mask_last(dg, raw, mode) == (rc, got)                 # may run again
                assert got == oracle_mask(raw, by_rec, mode)
                assert got == gpu(dg, raw, rows, mode)
                assert mask_last(dg, raw, mode)[0] == lib.E_ARG              # mask_fasta uploaded its own text
    raw = texts[1]
    dg.pred.predict_fasta(w, raw, 50, 256, True, 50, 50)
    assert mask_last(dg, raw, "soft", len(raw) - 1)[0] == lib.E_ARG      # another length
    assert mask_last(dg, raw, "soft")[0] == lib.OK
    dg.pred.predict_sequence(w, random_dna(5000, 3).encode(), 50, 256, True, 50, 50)
    assert mask_last(dg, raw, "soft")[0] == lib.E_ARG                    # an intervening call
    with pytest.raises(IndexError):
        dg.pred.predict_fasta(w, raw + b"\n\n>c\nACGT\n", 50, 256, True, 50, 50)
    assert mask_last(dg, raw + b"\n\n>c\nACGT\n", "soft")[0] == lib.E_ARG   # a failed call
    dg.pred.predict_fasta_tsv_sharded(w, raw, "f.fa", 50, 256, True, 50, 50, 0, 2)
    assert mask_last(dg, raw, "soft")[0] == lib.E_ARG                    # a sharded call


# ------------------------------------------------------------------ end to end through the CLI
def tsv_rows(tsv: bytes, headers):
    """{record: [(start, end)]} of a TSV text; headers: the kept records' headers (unique) in file order."""
    index = {h: r for r, h in enumerate(headers)}
    by_rec, total = {}, 0
    for line in tsv.decode().splitlines():
        _, h, s, e, _ = line.split("\t")
        by_rec.setdefault(index[h], []).append((int(s), int(e)))
        total += int(e) - int(s)
    return by_rec, total


def run_cli(tmp_path, mpath, fasta, extra=(), mask=None, mode="soft"):
    from deepgrp_b200.__main__ import CommandLineParser
    out = str(tmp_path / "out.tsv")
    argv = ["predict", mpath, fasta, "--output", out, *extra]
    if mask:
        argv += ["--mask", mask, "--mask_mode", mode]
    err = None
    try:
        CommandLineParser().parse_args(argv).run()
    except (IndexError, ValueError) as e:
        err = e
    with open(out, "rb") as fh:
        return fh.read(), err


def genome(rng, sizes, crlf_every=3):
    """Multi-record text: lowercase runs, N runs at the record edges, CRLF records, an empty-header record and a
    preamble.  -> (bytes, kept headers)."""
    parts, headers = ["; preamble\n"], []
    for i, n in enumerate(sizes):
        seq = np.frombuffer(random_dna(n, int(rng.integers(1 << 30))).encode(), np.uint8).copy()
        for _ in range(3):
            a = int(rng.integers(0, n))
            seq[a:a + int(rng.integers(1, 3000))] |= 32                             # lowercase run
        seq[:int(rng.integers(0, 80))] = ord("N")
        if n > 100:
            seq[n - int(rng.integers(0, 80)):] = ord("N")
        nl = "\r\n" if i % crlf_every == 1 else "\n"
        h = "" if i == 2 else "chr%d desc" % i
        if h:
            headers.append(h)
        s = seq.tobytes().decode()
        parts.append(">" + h + nl + nl.join(s[j:j + 60] for j in range(0, len(s), 60)) + nl)
    return "".join(parts).encode(), headers


@pytest.fixture(scope="module")
def model_path(dg, tmp_path_factory):
    p = str(tmp_path_factory.mktemp("m") / "w4.npz")
    dg.model.random_weights(150, 32, attention=True, seed=0).scaled(4.0).save_npz(p)
    return p


def check_cli(tmp_path, model_path, text, headers, extra=()):
    fa = str(tmp_path / "in.fa")
    with open(fa, "wb") as fh:
        fh.write(text)
    plain, err = run_cli(tmp_path, model_path, fa, extra)
    assert err is None
    by_rec, total = tsv_rows(plain, headers)
    assert total > 0
    for mode in MODES:
        mpath = str(tmp_path / ("masked.%s.fa" % mode))
        tsv, err = run_cli(tmp_path, model_path, fa, extra, mpath, mode)
        assert err is None
        assert tsv == plain
        with open(mpath, "rb") as fh:
            got = fh.read()
        assert got == oracle_mask(text, by_rec, mode)
        if mode == "hard":
            pos = positions(text)
            assert sum(len(pos[r][a:b]) for r, rr in by_rec.items() for a, b in rr) == total
            covered = np.zeros(len(text), bool)
            for r, rr in by_rec.items():
                for a, b in rr:
                    covered[pos[r][a:b]] = True
            g = np.frombuffer(got, np.uint8)
            assert int(covered.sum()) == total and (g[covered] == ord("N")).all()
    return plain


@pytest.mark.parametrize("extra", [(), ("--no_use_mss",)])
def test_cli_mask_end_to_end(dg, tmp_path, model_path, extra):
    rng = np.random.default_rng(11)
    text, headers = genome(rng, [int(x) for x in rng.integers(500, 60000, size=9)])
    check_cli(tmp_path, model_path, text, headers, extra)


def test_cli_mask_slices(dg, tmp_path, model_path):
    from deepgrp_b200.sharding import fasta_slices
    rng = np.random.default_rng(12)
    sizes = [10_000_000, 1000, 4_000_000, 2500, 7_000_000, 1200, 3_000_000, 800_000, 1000]
    text, headers = genome(rng, sizes)
    assert len(text) > 24 << 20
    assert len(fasta_slices(text, 1)[0]) - 1 >= 3
    check_cli(tmp_path, model_path, text, headers)


@pytest.mark.parametrize("kind", ["blank", "alln"])
def test_cli_mask_errors_in_the_second_slice(dg, tmp_path, model_path, kind):
    from deepgrp_b200.sharding import fasta_slices
    rng = np.random.default_rng(13)
    text, headers = genome(rng, [9_000_000, 5000, 3000, 200_000, 4000])
    cuts = fasta_slices(text, 1)[0]
    assert len(cuts) - 1 >= 2
    head, tail = text[:cuts[1]], text[cuts[1]:]
    lines_ = tail.split(b"\n")
    if kind == "blank":
        lines_.insert(len(lines_) // 2, b"")
    else:                                # a record of N only, in front of the slice's third record
        at = [i for i, x in enumerate(lines_) if x.startswith(b">")][2]
        lines_[at:at] = [b">allN", b"N" * 500]
    bad = head + b"\n".join(lines_)
    fa = str(tmp_path / "bad.fa")
    with open(fa, "wb") as fh:
        fh.write(bad)
    plain, err0 = run_cli(tmp_path, model_path, fa)
    mpath = str(tmp_path / "bad.masked.fa")
    tsv, err1 = run_cli(tmp_path, model_path, fa, (), mpath, "soft")
    want = IndexError if kind == "blank" else ValueError
    assert type(err0) is want and type(err1) is want
    assert tsv == plain
    kept_head = [h for h in headers if (">" + h).encode() in head]
    by_rec, _ = tsv_rows(b"".join(l + b"\n" for l in plain.splitlines() if l.split(b"\t")[1].decode() in kept_head),
                         kept_head)
    with open(mpath, "rb") as fh:
        assert fh.read() == oracle_mask(head, by_rec, "soft")


def test_cli_mask_refusals(tmp_path):
    from deepgrp_b200.__main__ import CommandLineParser
    for argv in (["predict", "m.npz", "x.fa", "--mask", "o.fa", "--stepwise"],
                 ["predict", "m.npz", "x.fa", "--mask", "-"]):
        with pytest.raises(SystemExit):
            CommandLineParser().parse_args(argv)
