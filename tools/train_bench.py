"""Training step time on one GPU: one JSON line for the default model shape (vecsize 342, units 60, attention, 5
classes) and batch 256.

    python tools/train_bench.py [--steps 50] [--warmup 10] [--oracle-steps 1]

Reports the median device time of a step (CUDA events around its phases: forward, head, BPTT, weight-gradient
reduction, update) and each phase's share of it, the median host wall time of a step (uploads of starts and masks,
the loss back), windows/s and positions/s, and -- for context only -- the time of the float64 CPU oracle
(oracle/train_oracle.py, torch autograd on the host cores) for one step on the same batch.  The record is 4 Mbp of
seeded random DNA with random annotations; nothing is written to disk."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deepgrp_b200 import _lib, model as dgmodel, training as dgtrain  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--vecsize", type=int, default=342)
    ap.add_argument("--units", type=int, default=60)
    ap.add_argument("--length", type=int, default=4_000_000)
    ap.add_argument("--oracle-steps", type=int, default=1, help="float64 CPU oracle steps to time (0: skip)")
    args = ap.parse_args(argv)
    T, U, B = args.vecsize, args.units, args.batch
    options = dgmodel.Options(vecsize=T, units=U, attention=True, batch_size=B, repeats_to_search=[1, 2, 3, 4])
    rng = np.random.default_rng(0)
    codes = rng.integers(0, 4, size=args.length).astype(np.uint8)
    y = np.zeros((5, args.length), np.int8)
    for c in range(1, 5):
        for a in rng.integers(0, args.length - 1000, size=args.length // 5000):
            y[c, a:a + int(rng.integers(50, 1000))] = 1
    y[0, ~y[1:].any(axis=0)] = 1
    model = dgmodel.create_model(options)
    ctx = _lib.context()
    tr = dgtrain.Trainer(model, options, ctx)
    tr.set_data(0, codes, dgtrain.labels_to_mask(y))
    sampler = dgtrain.BatchSampler(y, options)
    draws = [sampler.draw(rng) for _ in range(args.warmup + args.steps)]
    for d in draws[:args.warmup]:
        tr.step(d.starts, d.keep)
    wall, phases = [], []
    for d in draws[args.warmup:]:
        t0 = time.perf_counter()
        tr.step(d.starts, d.keep)
        wall.append((time.perf_counter() - t0) * 1e3)
        phases.append(list(tr.timings().values()))
    tr.close()
    phases = np.array(phases)
    device = phases.sum(axis=1)
    med = float(np.median(device))
    names = ("forward", "head", "bptt", "reduction", "update")
    result = dict(
        metric="train_step", gpu=gpu_info(), vecsize=T, units=U, attention=True, n_classes=5, batch=B,
        steps=args.steps, warmup=args.warmup,
        step_ms_device_median=round(med, 4),
        step_ms_device_min=round(float(device.min()), 4), step_ms_device_max=round(float(device.max()), 4),
        step_ms_wall_median=round(float(np.median(wall)), 4),
        windows_per_s=round(B / med * 1e3, 1), positions_per_s=round(B * T / med * 1e3, 1),
        phase_ms_median={n: round(float(np.median(phases[:, i])), 4) for i, n in enumerate(names)},
        phase_share={n: round(float(np.median(phases[:, i]) / med), 4) for i, n in enumerate(names)},
    )
    if args.oracle_steps > 0:
        from oracle import train_oracle
        import torch
        w = {k: (None if v is None else np.asarray(v, np.float64)) for k, v in model.as_dict().items()}
        times = []
        ymask = dgtrain.labels_to_mask(y)
        for d in draws[:args.oracle_steps]:
            t0 = time.perf_counter()
            train_oracle.train_loss_and_grads(w, codes, ymask, d.starts, d.keep, options.dropout, T)
            times.append(time.perf_counter() - t0)
        result["cpu_oracle_float64_step_s"] = round(float(np.median(times)), 3)
        result["cpu_oracle_threads"] = torch.get_num_threads()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
