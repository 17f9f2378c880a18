"""Cost of evaluation against a repeat annotation next to the prediction it scores, on one GPU.

Workload: the config-2 shape (vecsize 342, units 60, attention, random-init seed 0) on one 46.7 Mbp iid-ACGT record,
with 150 000 overlapping synthetic annotations of classes 1-4 (lengths 10-6000).  Times, each over --reps calls after
one warm-up call:
  predict        dgrp_predict_fasta on the record (host clock around the call, which ends in a device synchronise);
  evaluate       dgrp_evaluate_last on its rows (host clock: validation, host sort + merge + clip, upload, kernel,
                 copy back);
  eval_kernel    eval_confusion_kernel alone (CUDA events inside dgrp_evaluate_last);
  parse          preprocessing.read_annotation of the annotation written as a text file (host work, not in the ratio).
Prints the card's name and power limit from the same run and one JSON line.

    python tools/evaluate_bench.py [--reps 10] [--out FILE]
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

from deepgrp_b200 import _lib, model, preprocessing  # noqa: E402

L = 46_700_000
N_ANN = 150_000


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", str(_lib.default_device()), "--query-gpu=" + q, "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (v.strip() for v in out.split(","))))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    rng = np.random.default_rng(2)
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)]
    raw = b">chr21 synthetic\n" + np.concatenate([seq.reshape(-1, 100), np.full((L // 100, 1), 10, np.uint8)],
                                                 axis=1).tobytes()
    b = rng.integers(0, L, N_ANN)
    ann = np.stack([b, b + rng.integers(10, 6000, N_ANN), rng.integers(1, 5, N_ANN)], axis=1).astype(np.int64)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "ann.txt")
        np.savetxt(path, ann, fmt="chr21 %d %d %d RM")
        t0 = time.perf_counter()
        parsed = preprocessing.read_annotation(path, [1, 2, 3, 4])
        parse_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(parsed["chr21"], ann)

    w = model.random_weights(342, 60, attention=True, seed=0)
    ctx = _lib.context()
    C = w.n_classes
    ann_off = np.array([0, N_ANN], np.int64)
    counts = np.zeros((1, C, C), np.int64)
    buf = np.frombuffer(raw, np.uint8)
    n_rows, n_rec = ctypes.c_int64(0), ctypes.c_int64(0)

    def predict():
        _lib.check(_lib.lib().dgrp_predict_fasta(ctx.handle, w.device_handle(ctx), _lib.ptr(buf), len(raw), 50, 256,
                                                 1, 50, 50, _lib.COMPAT_REFERENCE, ctypes.byref(n_rows),
                                                 ctypes.byref(n_rec)))

    def evaluate():
        _lib.check(_lib.lib().dgrp_evaluate_last(ctx.handle, C, _lib.ptr(ann), _lib.ptr(ann_off), 1,
                                                 _lib.ptr(counts)))

    predict()
    evaluate()
    pred_ms, eval_ms, kern_ms = [], [], []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        predict()
        pred_ms.append((time.perf_counter() - t0) * 1e3)
    for _ in range(args.reps):
        t0 = time.perf_counter()
        evaluate()
        eval_ms.append((time.perf_counter() - t0) * 1e3)
        kern_ms.append(ctx.get_int("eval_kernel_ns") / 1e6)
    med = lambda v: float(np.median(v))                                     # noqa: E731
    res = {"workload": "config-2 shape, 46.7 Mbp record, %d annotations" % N_ANN, "card": card(),
           "reps": args.reps, "rows": int(n_rows.value), "predict_ms": med(pred_ms), "evaluate_ms": med(eval_ms),
           "eval_kernel_ms": med(kern_ms), "evaluate_over_predict": med(eval_ms) / med(pred_ms),
           "parse_annotation_ms": parse_ms, "predict_ms_all": pred_ms, "evaluate_ms_all": eval_ms,
           "eval_kernel_ms_all": kern_ms, "total_confusion": counts[0].tolist(),
           "TotalACC": float(np.trace(counts[0]) / counts[0].sum())}
    line = json.dumps(res)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    print("card: %s, power limit %s" % (res["card"].get("name"), res["card"].get("power.limit")))
    print(line)


if __name__ == "__main__":
    main()
