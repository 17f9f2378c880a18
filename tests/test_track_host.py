"""Probability tracks without a GPU: the kernel logic of csrc/track_core.cuh (the table dgrp_track_last builds, the bin
sums, the merge of equal bins and the line text, compiled for the host) byte for byte against an independent numpy
restatement of the bedGraph contract, and the `deepgrp predict --track` command line."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from deepgrp_b200 import __main__ as cli

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def restate_track(chrom, startpos, length, votes, bin):
    """The bedGraph lines of one record from the float32 votes of one class over its span [startpos, startpos + length):
    bins [k bin, (k + 1) bin) clipped to the span, s = float64 sum in position order (np.cumsum along each bin; zero
    padding in front of the span does not change a sequential sum), q = rint(s / n * 1000) (half to even), equal
    consecutive q merged, value "%d.%03d" % (q // 1000, q % 1000)."""
    votes = np.asarray(votes, np.float32)
    assert votes.shape == (length,)
    if length == 0:
        return b""
    k0, k1 = startpos // bin, (startpos + length - 1) // bin
    nb = k1 - k0 + 1
    pad = np.zeros(nb * bin, np.float64)
    off = startpos - k0 * bin
    pad[off:off + length] = votes.astype(np.float64)
    s = np.cumsum(pad.reshape(nb, bin), axis=1)[:, -1]
    k = np.arange(k0, k1 + 1, dtype=np.int64)
    starts = np.maximum(k * bin, startpos)
    ends = np.minimum((k + 1) * bin, startpos + length)
    q = np.rint(s / (ends - starts) * 1000.0).astype(np.int64)
    first = np.flatnonzero(np.r_[True, q[1:] != q[:-1]])
    last = np.r_[first[1:], nb] - 1
    return "".join("%s\t%d\t%d\t%d.%03d\n" % (chrom, a, b, v // 1000, v % 1000)
                   for a, b, v in zip(starts[first].tolist(), ends[last].tolist(), q[first].tolist())).encode()


@pytest.fixture(scope="module")
def host_track():
    so = os.path.join(HERE, "host", "libtrack_host.so")
    src = os.path.join(HERE, "host", "track_host.cpp")
    deps = [src] + [os.path.join(ROOT, "deepgrp_b200", "csrc", h) for h in ("track_core.cuh", "seg_core.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    lib = ctypes.CDLL(so)
    lib.track_host_text.restype = ctypes.c_int64
    lib.track_host_text.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 6 + \
        [ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]

    def text(C, cls, bin, records):
        """records: [(chrom, startpos, votes float32[length, C])] -> (bytes, number of lines)."""
        P = lambda a: ctypes.c_void_p(a.ctypes.data)            # noqa: E731
        pred = np.ascontiguousarray(np.concatenate([v for _, _, v in records] + [np.zeros((1, C), np.float32)]),
                                    dtype=np.float32)
        row_off = np.concatenate([[0], np.cumsum([len(v) for _, _, v in records])]).astype(np.int64)
        sp = np.array([s for _, s, _ in records] + [0], np.int64)
        ln = np.array([len(v) for _, _, v in records] + [0], np.int64)
        pfx = b"".join(c.encode() + b"\t" for c, _, _ in records) + b"\0"
        pbuf = np.frombuffer(pfx, np.uint8).copy()
        pfx_off = np.concatenate([[0], np.cumsum([len(c.encode()) + 1 for c, _, _ in records])]).astype(np.int64)
        lines = ctypes.c_int64(0)
        empty = np.zeros(1, np.uint8)
        need = lib.track_host_text(C, cls, bin, P(pred), P(row_off), P(sp), P(ln), P(pbuf), P(pfx_off),
                                   len(records), P(empty), 0, ctypes.byref(lines))
        out = np.zeros(max(need, 1), np.uint8)
        got = lib.track_host_text(C, cls, bin, P(pred), P(row_off), P(sp), P(ln), P(pbuf), P(pfx_off),
                                  len(records), P(out), need, ctypes.byref(lines))
        assert got == need
        return out[:need].tobytes(), lines.value
    return text


def votes(rng, length, C, levels=None):
    """Max-vote-like rows: runs of equal values (so that bins merge), some exact 0 and 1, and noise."""
    v = rng.random((length, C)).astype(np.float32)
    if levels is not None:
        v = np.asarray(levels, np.float32)[rng.integers(0, len(levels), (length, C))]
    if length == 0:
        return v
    runs = np.sort(rng.integers(0, length, size=min(length, 8)))
    for a, b in zip(runs[::2], runs[1::2]):
        v[a:b] = v[a]
    v[rng.integers(0, length, size=length // 10)] = 0.0
    v[rng.integers(0, length, size=length // 10)] = 1.0
    return v


def check(host_track, C, bin, records):
    for cls in range(1, C):
        got, n_lines = host_track(C, cls, bin, records)
        want = b"".join(restate_track(c, s, len(v), v[:, cls], bin) for c, s, v in records)
        assert got == want, (C, cls, bin)
        assert n_lines == want.count(b"\n")


@pytest.mark.parametrize("bin", [1, 7, 10, 1000, 10**6])
@pytest.mark.parametrize("C", [2, 5])
def test_kernel_logic_equals_restatement(host_track, C, bin):
    """Spans that start and end on and off bin boundaries, shorter than one bin, empty, and several records."""
    rng = np.random.default_rng(bin * 10 + C)
    records = []
    for i, (sp, length) in enumerate([(0, 1), (3, 5), (bin, bin), (bin - 1, 2), (17, 3 * bin + 4), (0, 0),
                                      (2 * bin + 1, max(bin - 2, 1)), (5, 2500), (bin * 3, 1)]):
        records.append(("chr%d" % i, sp, votes(rng, length, C)))
    check(host_track, C, bin, records)


@pytest.mark.parametrize("bin", [1, 2, 10])
def test_values_zero_one_and_ties(host_track, bin):
    """Bins whose mean is 0, 1 or exactly x.xxx5 (dyadic float32 votes): q rounds half to even."""
    C = 5
    levels = [0.0, 1.0, 0.0625, 0.1875, 0.3125, 0.4375, 0.5625, 0.9375, 0.125]
    rng = np.random.default_rng(bin)
    records = [("tie%d" % i, int(rng.integers(0, 30)), votes(rng, int(n), C, levels))
               for i, n in enumerate([1, 2, 9, 40, 333])]
    records.append(("zeros", 4, np.zeros((25, C), np.float32)))
    records.append(("ones", 0, np.ones((25, C), np.float32)))
    check(host_track, C, bin, records)
    one = [("t", 0, np.full((1, C), 0.0625, np.float32)), ("u", 0, np.full((1, C), 0.1875, np.float32))]
    assert host_track(C, 1, 1, one)[0] == b"t\t0\t1\t0.062\nu\t0\t1\t0.188\n"
    assert host_track(C, 2, 10, records[-2:])[0] == b"zeros\t4\t29\t0.000\nones\t0\t25\t1.000\n"


def test_lines_never_cross_records(host_track):
    """Two records with the same name and constant votes: one line each, and a line per bin change only."""
    C = 2
    same = np.full((30, C), 0.25, np.float32)
    got, n = host_track(C, 1, 10, [("c", 5, same), ("c", 0, same)])
    assert got == b"c\t5\t35\t0.250\nc\t0\t30\t0.250\n" and n == 2
    step = np.repeat(np.array([[0.5, 0.1], [0.5, 0.2], [0.5, 0.2]], np.float32), 10, axis=0)
    assert host_track(C, 1, 10, [("s", 0, step)])[0] == b"s\t0\t10\t0.100\ns\t10\t30\t0.200\n"


def test_large_coordinates(host_track):
    """Positions beyond 2^32 format with the 64-bit digit path."""
    C = 2
    sp = (1 << 33) + 3
    check(host_track, C, 1000, [("far", sp, votes(np.random.default_rng(1), 2100, C))])


# ---- command line -----------------------------------------------------------------------------------------
def parse(argv):
    return cli.CommandLineParser().parse_args(argv).args


def test_cli_parses_track():
    a = parse(["predict", "m.hdf5", "a.fa", "--output", "o.tsv", "--track", "out/t", "--track_bin", "333",
               "--mask", "m.fa"])
    assert (a.track, a.track_bin, a.mask) == ("out/t", 333, "m.fa")
    d = parse(["predict", "m.hdf5", "a.fa"])
    assert (d.track, d.track_bin) == (None, 10)
    r = parse(["-s", "30", "model.hdf5", "x.fa", "--track", "p"])
    assert (r.command, r.track) == ("predict", "p")
    assert parse(["predict", "m.hdf5", "a.fa", "--track", "p", "--track_bin", "1000000"]).track_bin == 10**6


@pytest.mark.parametrize("argv", [["--track", "p", "--stepwise"], ["--track", "-"], ["--track", "p", "--track_bin", "0"],
                                  ["--track_bin", "-3"], ["--track", "p", "--track_bin", "1000001"]])
def test_cli_refuses(argv, capsys):
    with pytest.raises(SystemExit) as e:
        parse(["predict", "m.hdf5", "a.fa"] + argv)
    assert e.value.code == 2
    assert "track" in capsys.readouterr().err
