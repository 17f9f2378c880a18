"""Cost of probability tracks (`deepgrp predict --track`) next to the prediction they come from, on one GPU.

Workload: the config-2 shape (vecsize 342, units 60, attention, random-init seed 0, 5 classes) on one 46.7 Mbp
iid-ACGT record.  Times, each over --reps calls after one warm-up call:
  predict / predict_keep   dgrp_predict_fasta without and with the keep_votes option, alternated (host clock around the
                           call, which ends in a device synchronise); append: the device time of the vote copy
                           (CUDA events, "votes_append_ns");
  track_b<N>               dgrp_track_last of every class 1-4 at bins 1 and 10 (host clock: table upload, kernels,
                           copy of the text to pinned memory); kernel: CUDA events from the first kernel to the last
                           ("track_kernel_ns", which includes the two waits for the line and byte counts);
  cli / cli_track          `deepgrp predict` on the record as a file, without and with --track (bin 10), alternated in
                           this process (host clock).
Bytes are what the kernels must move, computed from the shapes: the vote rows (20 B per base at 5 classes: the bin
kernel reads one column, but 4-byte columns 20 bytes apart pull every 32-byte sector), the bin words (written once,
read by the flag count and by the compaction, and twice per line), the line starts and the text.
Prints the card's name and power limit from the same run and one JSON line.

    python tools/track_bench.py [--reps 5] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from deepgrp_b200 import _lib, model  # noqa: E402
from deepgrp_b200.__main__ import CommandLineParser  # noqa: E402

L = 46_700_000
HBM = 7.7e12


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", str(_lib.default_device()), "--query-gpu=" + q, "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (v.strip() for v in out.split(","))))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    rng = np.random.default_rng(2)
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)]
    raw = b">chr21 synthetic\n" + np.concatenate([seq.reshape(-1, 100), np.full((L // 100, 1), 10, np.uint8)],
                                                 axis=1).tobytes()
    w = model.random_weights(342, 60, attention=True, seed=0)
    ctx = _lib.context()
    C = w.n_classes
    buf = np.frombuffer(raw, np.uint8)
    n_rows, n_rec = ctypes.c_int64(0), ctypes.c_int64(0)
    med = lambda v: float(np.median(v))                                     # noqa: E731

    def predict(keep):
        ctx.set_int("keep_votes", keep)
        try:
            t0 = time.perf_counter()
            _lib.check(_lib.lib().dgrp_predict_fasta(ctx.handle, w.device_handle(ctx), _lib.ptr(buf), len(raw), 50,
                                                     256, 1, 50, 50, _lib.COMPAT_REFERENCE, ctypes.byref(n_rows),
                                                     ctypes.byref(n_rec)))
            return (time.perf_counter() - t0) * 1e3
        finally:
            ctx.set_int("keep_votes", 0)

    predict(0)
    predict(1)
    res = {"workload": "config-2 shape, one 46.7 Mbp record, 5 classes", "card": card(), "reps": args.reps}
    p0, p1, app = [], [], []
    for _ in range(args.reps):
        p0.append(predict(0))
        p1.append(predict(1))
        app.append(ctx.get_int("votes_append_ns") / 1e6)
    vote_bytes = L * C * 4
    res.update(predict_ms=med(p0), predict_keep_ms=med(p1), append_ms=med(app), predict_ms_all=p0,
               predict_keep_ms_all=p1, append_ms_all=app,
               append_hbm_share=2 * vote_bytes / HBM / (med(app) / 1e3))   # read + write
    text, n = ctypes.c_void_p(), ctypes.c_int64(0)
    for bin in (1, 10):
        bins = -(-L // bin)
        for cls in range(1, C):                                              # warm-up
            _lib.check(_lib.lib().dgrp_track_last(ctx.handle, cls, bin, ctypes.byref(text), ctypes.byref(n)))
        _lib.check(_lib.lib().dgrp_track_last(ctx.handle, 1, bin, ctypes.byref(text), ctypes.byref(n)))
        n_lines = ctypes.string_at(text.value, n.value).count(b"\n")
        wall, kern, nbytes = [], [], []
        for _ in range(args.reps):
            for cls in range(1, C):
                t0 = time.perf_counter()
                _lib.check(_lib.lib().dgrp_track_last(ctx.handle, cls, bin, ctypes.byref(text), ctypes.byref(n)))
                wall.append((time.perf_counter() - t0) * 1e3)
                kern.append(ctx.get_int("track_kernel_ns") / 1e6)
                nbytes.append(int(n.value))
        moved = vote_bytes + bins * 4 * 3 + n_lines * (2 * 4 + 2 * 8) + med(nbytes)
        res["track_b%d" % bin] = {"bins": bins, "lines_class1": n_lines, "text_bytes_median": med(nbytes),
                                  "call_ms": med(wall), "kernel_ms": med(kern), "bytes_moved": moved,
                                  "kernel_hbm_share": moved / HBM / (med(kern) / 1e3),
                                  "call_ms_all": wall, "kernel_ms_all": kern}
    with tempfile.TemporaryDirectory() as tmp:
        fa, mp = os.path.join(tmp, "r.fa"), os.path.join(tmp, "m.npz")
        with open(fa, "wb") as fh:
            fh.write(raw)
        w.save_npz(mp)
        cli = {"plain": [], "track": []}
        base = ["predict", mp, fa, "--output", os.path.join(tmp, "o.tsv")]
        CommandLineParser().parse_args(base).run()                           # warm-up
        for _ in range(args.reps):
            for kind, extra in (("plain", []), ("track", ["--track", os.path.join(tmp, "t")])):
                t0 = time.perf_counter()
                CommandLineParser().parse_args(base + extra).run()
                cli[kind].append((time.perf_counter() - t0) * 1e3)
        res.update(cli_ms=med(cli["plain"]), cli_track_ms=med(cli["track"]), cli_ms_all=cli["plain"],
                   cli_track_ms_all=cli["track"],
                   track_file_bytes=sum(os.path.getsize(os.path.join(tmp, "t.%d.bedGraph" % c)) for c in range(1, C)))
    line = json.dumps(res)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    print("card: %s, power limit %s" % (res["card"].get("name"), res["card"].get("power.limit")))
    print(line)


if __name__ == "__main__":
    main()
