"""Repeat masking on one GPU: device time of the mask kernels and end-to-end `deepgrp predict --mask` against the
default route.

Input: a seeded synthetic genome-shaped FASTA (records of 1 kb to 40 Mbp, 60-column lines, lowercase and N runs),
about 400 MB by default, which is larger than the 126 MB of L2, written to a temporary directory.

1. Kernels: `dgrp_mask_fasta` with seeded rows covering about half of the positions, warmed up, then `--passes`
   calls under torch.profiler; the device time of every kernel the call launches is summed by name.  The bytes
   the mask needs are counted from the sizes: the classification reads the text twice (tile functions, counts),
   the paint writes one bit per position and the mask kernel reads the text and the bitmap and writes the text.
2. End to end: `python -m deepgrp_b200 predict` on the file, with and without `--mask`, alternated, wall clock.

Prints one JSON object; `--json PATH` also writes it to PATH.
Usage: python tools/mask_bench.py [--mbytes 400] [--passes 20] [--e2e 2] [--json PATH]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_TBS = 7.7      # HBM3e bandwidth of one B200 (data sheet)


def synthetic_genome(nbytes: int, seed: int = 0) -> bytes:
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b"ACGT", np.uint8)
    parts, total, i = [], 0, 0
    while total < nbytes:
        n = int(min(10 ** rng.uniform(3, 7.6), max(nbytes - total, 1000)))
        seq = lut[rng.integers(0, 4, size=n)]
        for _ in range(max(1, n // 200000)):
            a = int(rng.integers(0, n))
            seq[a:a + int(rng.integers(100, 20000))] |= 32
            b = int(rng.integers(0, n))
            seq[b:b + int(rng.integers(10, 5000))] = ord("N")
        full = n // 60 * 60
        body = np.concatenate([seq[:full].reshape(-1, 60), np.full((full // 60, 1), 10, np.uint8)], axis=1).ravel()
        tail = seq[full:].tobytes() + (b"\n" if n > full else b"")
        rec = b">chr%d synthetic\n" % i + body.tobytes() + tail
        parts.append(rec)
        total += len(rec)
        i += 1
    return b"".join(parts)


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = (x.strip() for x in out.split(","))
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:                       # noqa: BLE001
        return {"gpu": "unknown (%s)" % e}


def kernel_times(raw: bytes, passes: int) -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile
    from deepgrp_b200 import _lib, prediction
    # rows: every kept record, seeded disjoint rows over about half of its positions
    ctx = _lib.context()
    buf = np.frombuffer(raw, np.uint8)
    heads = np.flatnonzero(buf == ord(">"))
    ends = np.append(heads[1:], len(buf))
    rng = np.random.default_rng(1)
    rows = []
    for r, (h, e) in enumerate(zip(heads, ends)):
        nl = int(np.argmax(buf[h:e] == 10))
        n = int(np.count_nonzero(buf[h + nl:e] != 10))
        cuts = np.unique(rng.integers(0, n, size=max(2, n // 400)))
        rows += [(int(a), int(b), 1, r) for a, b in zip(cuts[0::2], cuts[1::2]) if a < b]
    rows = np.array(rows, dtype=_lib.ROW_DTYPE)
    covered = int((rows["end"] - rows["start"]).sum())
    for _ in range(3):
        prediction.mask_fasta(raw, rows, "soft")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(passes):
            prediction.mask_fasta(raw, rows, "soft")
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and "kernel" in ev.name:
            key = ev.name.split("(")[0].replace("void ", "").replace("dgrp::", "")
            per[key] = per.get(key, 0.0) + ev.device_time / 1e3 / passes        # ms per call
    ctx.synchronize()
    n = len(raw)
    n_seq = int(np.count_nonzero((buf != 10)) - sum(int(np.argmax(buf[h:e] == 10)) for h, e in zip(heads, ends)))
    classify_ms = sum(v for k, v in per.items() if k.startswith(("fa_tile", "fa_count", "cp_scan")))
    mask_ms = per.get("mask_paint_kernel", 0.0) + per.get("fa_mask_kernel", 0.0)
    mask_bytes = 2 * n + 2 * (n_seq // 8) + rows.nbytes
    classify_bytes = 2 * n
    return {
        "bytes": n, "positions": n_seq, "rows": int(rows.size), "covered": covered, "passes": passes,
        "kernels_ms": {k: round(v, 4) for k, v in sorted(per.items())},
        "paint_plus_mask_ms": round(mask_ms, 4),
        "paint_plus_mask_GBs": round(mask_bytes / mask_ms / 1e6, 1) if mask_ms else None,
        "paint_plus_mask_share_of_hbm": round(mask_bytes / mask_ms / 1e6 / (HBM_TBS * 1e3), 3) if mask_ms else None,
        "classify_ms": round(classify_ms, 4),
        "all_mask_kernels_ms": round(mask_ms + classify_ms, 4),
        "all_mask_kernels_share_of_hbm": round((mask_bytes + classify_bytes) / (mask_ms + classify_ms) / 1e6
                                               / (HBM_TBS * 1e3), 3) if mask_ms else None,
    }


def end_to_end(path: str, model: str, reps: int, tmp: str) -> dict:
    times = {"default": [], "mask": []}
    for _ in range(reps):
        for kind in ("default", "mask"):
            cmd = [sys.executable, "-m", "deepgrp_b200", "predict", model, path, "--output", os.path.join(tmp, "o.tsv")]
            if kind == "mask":
                cmd += ["--mask", os.path.join(tmp, "masked.fa")]
            t0 = time.perf_counter()
            subprocess.run(cmd, check=True, cwd=ROOT)
            times[kind].append(time.perf_counter() - t0)
    with open(os.path.join(tmp, "o.tsv"), "rb") as fh:
        n_rows = fh.read().count(b"\n")
    return {"rows": n_rows, "default_s": [round(x, 3) for x in times["default"]],
            "mask_s": [round(x, 3) for x in times["mask"]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mbytes", type=int, default=400)
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--e2e", type=int, default=2, help="end-to-end repetitions of each route (0: skip)")
    ap.add_argument("--json", type=str, default=None, help="also write the result to this file")
    args = ap.parse_args()
    from deepgrp_b200 import model as dgmodel
    res = gpu_info()
    with tempfile.TemporaryDirectory() as tmp:
        raw = synthetic_genome(args.mbytes << 20)
        path = os.path.join(tmp, "genome.fa")
        with open(path, "wb") as fh:
            fh.write(raw)
        res["kernels"] = kernel_times(raw, args.passes)
        if args.e2e:
            mpath = os.path.join(tmp, "w.npz")
            dgmodel.random_weights(150, 32, attention=True, seed=0).save_npz(mpath)
            res["end_to_end"] = end_to_end(path, mpath, args.e2e, tmp)
    text = json.dumps(res)
    print(text)
    if args.json:
        with open(args.json, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
