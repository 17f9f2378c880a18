#!/usr/bin/env python
"""bench.py -- bases classified per second (Mbp/s) on the DeepGRP prediction hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mbp M] [--dump-outputs DIR]

One "step" = one pass of the whole hot path (forward + vote + score + MSS + segment extraction)
over one synthetic record.  Workload at N=1: BASELINE.json configs[1] -- defaults.toml architecture
(vecsize 342, units 60, attention), random-init weights (seed 0), one 46.7 Mbp iid-ACGT record.
With N ranks every rank processes its own record of that size (contig sharding, no collective on
the data path), so `scaling` is "weak" and `value` = N * bases / max-over-ranks time.

Keys beyond the base contract:
  value      device-resident: base codes already in HBM, timed with CUDA events on the library's
             stream (exposed as a torch ExternalStream), L2 flushed between steps;
  e2e        the same metric through the public API `deepgrp_b200.prediction.predict_fasta_tsv`
             with the FASTA text in pinned HOST memory: H2D of the text, GPU decode, forward,
             MSS, D2H of the rows and TSV formatting all inside the timed region;
  roofline   the dominant kernel (the fused GRU/attention/vote kernel): algorithmic FLOPs
             (12TU^2 + 85TU + 3T per window, BASELINE.md section 3) / its CUDA-event time, against the
             measured bf16 tensor peak of MEASURED_PEAKS.json;
  cpu_baseline  the oracle port (reference restated on CPU, TF absent) on a bounded prefix.
`--impl reference` times the CPU restatement of the reference path only (rank 0).
`--dump-outputs DIR` writes what the last timed `value` step computed on rank 0 (see dump_outputs); the inputs
depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_DEFAULT, U_DEFAULT = 342, 60          # defaults.toml
STEP, BATCH, MIN_MSS, XDROP = 50, 256, 50, 50
CONFIG2_BASES = 46_700_000


def synth_codes(n, seed):
    """iid uniform ACGT codes (SURVEY.md section 8d: default_rng([1, k]))."""
    rng = np.random.default_rng(seed)
    return rng.integers(0, 4, size=n, dtype=np.uint8)


def fasta_text(codes, header, width=60):
    """FASTA text (bytes) of one record, `width` columns per line."""
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    n = letters.size
    full = n // width
    body = np.empty((full, width + 1), dtype=np.uint8)
    body[:, :width] = letters[:full * width].reshape(full, width)
    body[:, width] = ord("\n")
    tail = letters[full * width:].tobytes()
    return b">" + header.encode() + b"\n" + body.tobytes() + (tail + b"\n" if tail else b"")


def flops_per_window(T, U, rnn="GRU"):
    """Algorithmic FLOPs of one window (BASELINE.md section 3): recurrent product of both passes, input
    projection (dense-equivalent), attention, FF.  LSTM (4 gates, no attention, FF on U features)."""
    if rnn == "LSTM":
        return 16 * T * U * U + 80 * T * U + 10 * T * U
    return 12 * T * U * U + 85 * T * U + 3 * T


FORWARD_KERNELS = {
    0: "gru_attention_vote_kernel (fp32 FFMA)",
    1: "gru_tc_attention_vote_kernel (tcgen05, two tiles per SM, fp16 x2 operand pieces)",
    2: "rnn_tcw_kernel (tcgen05, one tile per SM, N-split MMAs, fp16 x2 operand pieces)",
    3: "rnn_tcw_kernel (tcgen05 cta_group::2, one tile per SM of a CTA pair, fp16 x2 operand pieces)",
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md).  Started before
    the warm-up (nvidia-smi needs ~0.2 s to come up); only the samples that arrive between mark_begin()
    and stop() count."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.t_begin = None

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                 "-lms", "40"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.perf_counter() + 0.05   # the row in flight when the region ended
        time.sleep(0.1)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = self.t_begin if self.t_begin is not None else 0.0
        for ts, r in self.rows:
            if ts < t0 or ts > t_end:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        # under load = samples in the upper half of the observed range
        load = [v for v in sm if v >= 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(load)) if load else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_weights(args):
    """Random-init weights of the requested architecture (Keras initialisers, seed 0), optionally scaled
    (SURVEY.md section 8d: the x4 set has confident outputs, so K6-K8 and the TSV see realistic dynamics)."""
    from deepgrp_b200 import model
    w = model.random_weights(args.vecsize, args.units, attention=True, seed=0, rnn=args.rnn)
    return w.scaled(args.weight_scale) if args.weight_scale != 1.0 else w


def host_threads():
    """Host cores this process may run on (affinity-aware)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return p["bf16_tflops_sustained"], p["hbm_gbs"], "measured"
    except (OSError, KeyError, ValueError):
        return 1400.0, 6650.0, "fallback"


def ncu_traffic(args):
    """dram__bytes_read.sum + dram__bytes_write.sum of the forward kernel, per launch, from the committed
    `ncu --set full` capture of this same workload (profiles/r02v_*); None for any other workload."""
    if (args.bases, args.vecsize, args.units) != (CONFIG2_BASES, T_DEFAULT, U_DEFAULT):
        return None
    try:
        import csv
        rows = list(csv.reader(open(os.path.join(ROOT, "profiles", "r02v_fwd_tc_ncu_raw.csv"))))
        col = {name: (unit, val) for name, unit, val in zip(rows[0], rows[1], rows[2])}
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        total = 0.0
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            unit, val = col[key]
            total += float(val) * scale[unit]
        return total
    except (OSError, KeyError, ValueError, IndexError):
        return None


def cpu_reference_step(codes_prefix, weights, T, threads):
    """The reference path restated on CPU (oracle port; TF absent): encode, windows, forward
    (torch.nn.GRU engine), max-vote incl. the partial-batch placement, MSS, segments, TSV."""
    from oracle import oracle as orc
    import torch
    torch.set_num_threads(threads)
    text = fasta_text(codes_prefix, "synthetic_prefix")
    with tempfile.NamedTemporaryFile("wb", suffix=".fa", delete=False) as fh:
        fh.write(text)
        path = fh.name
    try:
        t0 = time.perf_counter()
        tsv = orc.predict_fasta_tsv(path, weights.as_dict(), T, BATCH, STEP, True, MIN_MSS, XDROP,
                                    engine="torch")
        dt = time.perf_counter() - t0
    finally:
        os.unlink(path)
    return dt, len(tsv)


def run_reference(args, rank, world):
    if rank != 0:
        return
    from deepgrp_b200 import model
    weights = make_weights(args)
    threads = host_threads()
    sample = args.ref_bases
    codes = synth_codes(sample, [1, 0])
    for _ in range(args.warmup):
        cpu_reference_step(codes[:max(args.vecsize * 4, sample // 10)], weights, args.vecsize, threads)
    times = [cpu_reference_step(codes, weights, args.vecsize, threads)[0] for _ in range(args.steps)]
    total = sum(times)
    per_step = sorted(sample / t / 1e6 for t in times)
    value = sample * args.steps / total / 1e6
    line = {
        "impl": "reference", "metric": "bases classified/sec (Mbp/s), FASTA file -> TSV text on the host CPU", "value": value,
        "unit": "Mbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, sample),
        "cpu_baseline": {"value": value, "unit": "Mbp/s", "cores": threads, "kind": "port",
                         "min": per_step[0], "median": per_step[len(per_step) // 2], "max": per_step[-1],
                         "sample": "%d-base prefix of the workload per step (%d bases over the timed steps; the "
                                   "path is linear in the record length); reference restated on CPU "
                                   "(TF absent): oracle port with torch.nn.GRU engine"
                                   % (sample, sample * args.steps)},
        "e2e": {"value": value, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_name(args):
    """Which BASELINE.json configuration the arguments describe (the default run is configs[1])."""
    shape = (args.vecsize, args.units)
    if shape == (T_DEFAULT, U_DEFAULT):
        arch = "defaults.toml architecture"
        which = "configs[1]" if args.bases == CONFIG2_BASES else ("configs[2]" if args.bases == 248_000_000 else
                                                                  "configs[1] at another record length")
    elif shape == (150, 32):
        arch, which = "tests/test_model.json architecture", "configs[0]"
    elif shape in ((260, 50), (512, 128)):
        arch = "hyperopt search-space point 5%s (SURVEY.md section 8d)" % ("a" if shape == (260, 50) else "b")
        which = "configs[4]"
    else:
        return "custom workload, not a BASELINE.json configuration (vecsize %d, units %d, attention)" % shape
    return "BASELINE.json %s: %s (vecsize %d, units %d, attention)" % (which, arch, args.vecsize, args.units)


def workload_config(args, bases):
    return {"workload": workload_name(args) + ", random-init weights seed 0, synthetic iid-ACGT single-record FASTA",
            "bases_per_record": int(bases), "step_size": STEP, "batch_size": BATCH,
            "min_mss_len": MIN_MSS, "xdrop_len": XDROP, "compat": "reference",
            "l2": "flushed between steps (256 MiB memset); per-step working set (predictions + "
                  "scratch, >1.5 GB) also exceeds L2",
            "sharding": "one record per rank, no collective"}


DUMP_LABELS, DUMP_ROWS = 4_000_000, 1_000_000     # at most 16 MB of labels and 24 MB of rows


def dump_outputs(out_dir, ctx, length, n_rows):
    """What the last dgrp_predict_codes_dev left on the device, as float .npy files in `out_dir`: labels.npy, the
    final labels (float32) at DUMP_LABELS positions; label_counts.npy, the count of each label over all positions
    (float64); rows.npy, DUMP_ROWS of the rows as (start, end, label) (float64).  Positions and rows are fixed
    samples (seeded, sorted) when there are more; all of them otherwise."""
    from deepgrp_b200 import _lib
    labels = np.empty(length, dtype=np.uint8)
    rows = np.empty((n_rows, 3), dtype=np.int64)
    _lib.check(_lib.lib().dgrp_predict_codes_dev_results(ctx.handle, _lib.ptr(labels), length, _lib.ptr(rows),
                                                         n_rows))

    def sample(n, k, seed):
        return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "labels.npy"), labels[sample(length, DUMP_LABELS, 0)].astype(np.float32))
    np.save(os.path.join(out_dir, "label_counts.npy"), np.bincount(labels, minlength=5).astype(np.float64))
    np.save(os.path.join(out_dir, "rows.npy"), rows[sample(n_rows, DUMP_ROWS, 1)].astype(np.float64))


def numa_bind(local_rank):
    """Run this rank (and what it allocates: first touch decides where pinned buffers live) on the CPUs local to
    its GPU, as `numactl --cpunodebind` would.  Returns a short description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (dom, bus, dev)
        cpus = set()
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return "%d cpus local to GPU %d" % (len(allowed), local_rank)
    except (OSError, ValueError, AttributeError, RuntimeError):
        pass
    return "not bound"


def run_ours(args, rank, world, local_rank):
    import ctypes
    import torch
    import torch.distributed as dist
    from deepgrp_b200 import _lib, prediction

    torch.cuda.set_device(local_rank)
    binding = numa_bind(local_rank) if args.numa_bind else "not bound"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.context(local_rank)
    ctx.set_int("stream_early_rows", args.early_rows)
    ctx.set_int("stream_early_slabs", args.early_slabs)
    ctx.set_int("stream_early_ratio", args.early_ratio)
    if args.mss_chunk:
        ctx.set_int("mss_chunk", args.mss_chunk)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    devnull = open(os.devnull, "wb")
    sections = set(args.sections.split(","))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(values):
        t = torch.tensor(values, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.cpu()]

    def measure(weights, L, steps, warmup, sample_clocks, dump_dir=None):
        """One record of L bases per rank: `value` leg (codes resident in HBM, CUDA events on the library's
        stream) and `e2e` leg (FASTA text in pinned host memory -> TSV text on the host, through the public
        streaming API, wall clock).  With `dump_dir`, rank 0 writes the last `value` step's outputs there."""
        handle = weights.device_handle(ctx)
        codes = synth_codes(L, [1, rank])
        d_codes = torch.from_numpy(codes).cuda()
        text = fasta_text(codes, "synthetic_%dbp_rank%d" % (L, rank))
        pinned = torch.empty(len(text), dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = np.frombuffer(text, dtype=np.uint8)
        raw_view = pinned.numpy()
        n_rows = ctypes.c_int64(0)

        def device_step():
            with torch.cuda.stream(stream):
                flush.zero_()
            _lib.check(_lib.lib().dgrp_predict_codes_dev(
                ctx.handle, handle, ctypes.c_void_p(d_codes.data_ptr()), L, STEP, BATCH, 1, MIN_MSS, XDROP,
                _lib.COMPAT_REFERENCE, ctypes.byref(n_rows)))
            return ctx.timings()

        def e2e_step():
            if args.e2e_api == "oneshot":   # the one-call form (whole TSV in one pinned buffer, one D2H copy)
                view = prediction.predict_fasta_tsv_view(weights, raw_view, "synthetic.fa", STEP, BATCH, True,
                                                         MIN_MSS, XDROP)
                devnull.write(view)
                return {"h2d_bytes": len(text), "d2h_bytes": len(view)}
            return prediction.predict_fasta_tsv_stream(weights, raw_view, "synthetic.fa", devnull, STEP, BATCH,
                                                       True, MIN_MSS, XDROP)

        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        t_w = time.perf_counter()
        for _ in range(warmup):
            device_step()
        barrier()
        print("[bench] rank %d: %d warm-up steps in %.2f s" % (rank, warmup, time.perf_counter() - t_w),
              file=sys.stderr, flush=True)
        launches0 = ctx.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage_ms = []
        barrier()
        if sampler:
            sampler.mark_begin()
        ev0.record(stream)
        for _ in range(steps):
            stage_ms.append(device_step())
        ev1.record(stream)
        barrier()
        elapsed_ms = ev0.elapsed_time(ev1)
        launches = ctx.launch_count() - launches0
        clocks = sampler.stop() if sampler else None
        used_kernel = ctx.get_int("forward_used_tc")
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, ctx, L, int(n_rows.value))
        for _ in range(max(1, min(warmup, 2))):
            st = e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            st = e2e_step()
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        elapsed_ms, e2e_ms = allmax([elapsed_ms, e2e_ms])
        mean_stage = {k: float(np.mean([x[k] for x in stage_ms]))
                      for k in ("forward_ms", "score_ms", "mss_ms", "segments_ms", "total_ms")}
        return {"value": world * L * steps / (elapsed_ms / 1e3) / 1e6, "ms_per_step": elapsed_ms / steps,
                "e2e_value": world * L * steps / (e2e_ms / 1e3) / 1e6, "e2e_ms_per_step": e2e_ms / steps,
                "h2d": st["h2d_bytes"], "d2h": st["d2h_bytes"], "rows": int(n_rows.value), "launches": int(launches),
                "stages_ms": mean_stage, "clocks": clocks, "kernel": used_kernel, "codes": codes,
                "mss_rounds": ctx.get_int("mss_rounds"), "early_parts": ctx.get_int("stream_early_parts"),
                "e2e_last": {k: st[k] for k in ("forward_ms", "gpu_ms", "launches", "waits_ms") if k in st}}

    weights = make_weights(args)
    L = args.bases
    main = measure(weights, L, args.steps, args.warmup, True, args.dump_outputs)
    tflops_peak, hbm_peak, peak_kind = peaks()
    n_windows = len(range(0, L - args.vecsize, STEP))
    kernel_ms = main["stages_ms"]["forward_ms"]
    achieved = flops_per_window(args.vecsize, args.units, args.rnn) * n_windows / (kernel_ms / 1e3) / 1e12
    line = {
        "metric": "bases classified/sec (Mbp/s): value = record resident in HBM (device-timed); e2e = FASTA text in "
                  "host memory -> TSV text in host memory",
        "value": main["value"], "unit": "Mbp/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, L),
        "clocks": main["clocks"],
        "e2e": {"value": main["e2e_value"], "unit": "Mbp/s", "h2d_bytes_per_step": main["h2d"],
                "d2h_bytes_per_step": main["d2h"], "ms_per_step": main["e2e_ms_per_step"],
                "api": "deepgrp_b200.prediction.predict_fasta_tsv_stream (C ABI dgrp_fasta_stream_*)",
                "early_parts": main["early_parts"], "last_step": main["e2e_last"]},
        "gpu_launches": main["launches"],
        "roofline": {"bound": "tensor", "kernel": FORWARD_KERNELS[main["kernel"]],
                     "achieved": achieved, "peak": tflops_peak, "unit": "TFLOP/s",
                     "frac": achieved / tflops_peak, "traffic": ncu_traffic(args),
                     "traffic_unit": "bytes of DRAM read + written per launch (ncu --set full, profiles/)",
                     "peak_kind": peak_kind,
                     "kernel_ms": kernel_ms, "share_of_step": kernel_ms / main["ms_per_step"]},
        "stages_ms": main["stages_ms"], "rows_per_step": main["rows"], "mss_rounds": main["mss_rounds"],
        "numa": binding,
    }
    # -- the confident-output weight set (SURVEY.md section 8d): same shapes, weights x 4 ------------------------
    if "x4" in sections and args.weight_scale == 1.0:
        args4 = argparse.Namespace(**vars(args))
        args4.weight_scale = 4.0
        x4 = measure(make_weights(args4), L, min(args.steps, 5), 2, False)
        line["x4"] = {"weights": "the same random-init weights x 4 (max probability up to 0.9, all classes present)",
                      "value": x4["value"], "ms_per_step": x4["ms_per_step"], "e2e": x4["e2e_value"],
                      "e2e_ms_per_step": x4["e2e_ms_per_step"], "e2e_early_parts": x4["early_parts"],
                      "rows_per_step": x4["rows"],
                      "d2h_bytes_per_step": x4["d2h"], "stages_ms": x4["stages_ms"], "unit": "Mbp/s"}
    # -- BASELINE.json configs[2]: ONE chr1-sized record split by position over the ranks (strong scaling) -------
    if "strong" in sections:
        a3 = argparse.Namespace(**vars(args))
        a3.bases, a3.steps, a3.warmup = args.strong_bases, min(args.steps, 3), 1
        strong = chunk_sharded(a3, rank, world, local_rank, ctx, stream, flush)
        if rank == 0:
            line["strong"] = strong
    # -- BASELINE.json configs[4]: the widest search-space point (T = 512, U = 128) on a 248 Mbp record, chunk-sharded ------
    if "config5b" in sections:
        a5 = argparse.Namespace(**vars(args))
        a5.bases, a5.vecsize, a5.units, a5.steps, a5.warmup = args.strong_bases, 512, 128, min(args.steps, 2), 1
        c5 = chunk_sharded(a5, rank, world, local_rank, ctx, stream, flush)
        if rank == 0:
            nw = len(range(0, a5.bases - a5.vecsize, STEP))
            tf = flops_per_window(a5.vecsize, a5.units) * nw / world / (c5["stages_ms"]["range_forward_score_max_over_ranks"] / 1e3) / 1e12
            c5["roofline"] = {"bound": "tensor", "kernel": FORWARD_KERNELS[ctx.get_int("forward_used_tc")],
                              "achieved_per_gpu": tf, "peak": tflops_peak, "unit": "TFLOP/s", "frac": tf / tflops_peak,
                              "note": "forward + vote + score time of the slowest rank; algorithmic FLOPs of its share"}
            line["config5b"] = c5
    # -- BASELINE.json configs[3]: the multi-FASTA genome, contig-sharded, end to end ------------------------------
    if "genome" in sections:
        g = genome_section(args, rank, world, weights, devnull, barrier)
        if rank == 0:
            line["genome"] = g
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        sample = min(args.ref_bases // 3, L)
        vals = []
        for k in range(3):
            dt, _ = cpu_reference_step(main["codes"][k * sample:(k + 1) * sample], weights, args.vecsize, threads)
            vals.append(sample / dt / 1e6)
        line["cpu_baseline"] = {
            "value": float(np.median(vals)), "min": min(vals), "max": max(vals), "unit": "Mbp/s", "cores": threads,
            "kind": "port",
            "sample": "3 disjoint %d-base pieces of the workload, median; reference restated on CPU (TF absent): "
                      "oracle port with torch.nn.GRU engine" % sample}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def genome_section(args, rank, world, weights, devnull, barrier):
    """BASELINE.json configs[3] in shape, scaled to the number of ranks (world / 8 of the 3.1 Gbp genome, so the
    work per GPU is that of the 8-GPU target run): rank 0 writes the multi-FASTA into /dev/shm, every rank maps it
    and streams its own contigs (host header index, largest slice first) through the pipelined public API."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import genome_bench
    from deepgrp_b200 import prediction
    scale = args.genome_scale if args.genome_scale > 0 else world / 8.0
    path = "/dev/shm/dgrp_config4_%d.npy" % os.getpid() if world == 1 else "/dev/shm/dgrp_config4_shared.npy"
    t_gen = time.perf_counter()
    if rank == 0:
        bases = genome_bench.write_fasta(path, scale)
        json.dump({"bases": bases}, open(path + ".json", "w"))
    barrier()
    t_gen = time.perf_counter() - t_gen
    bases = json.load(open(path + ".json"))["bases"]
    raw = np.load(path, mmap_mode="r")

    def step():
        return prediction.predict_fasta_tsv_stream(weights, raw, "genome.fa", devnull, STEP, BATCH, True, MIN_MSS,
                                                   XDROP, rank=rank, world=world)
    step()                                    # warm-up: buffers, first touch of the mapped file
    walls, locals_ = [], []
    for _ in range(2):
        barrier()
        t0 = time.perf_counter()
        st = step()
        locals_.append(time.perf_counter() - t0)
        barrier()
        walls.append(time.perf_counter() - t0)
    stats = torch.tensor([float(st["d2h_bytes"]), float(st["rows"]), min(locals_), float(st["h2d_bytes"]),
                          st["forward_ms"] / 1e3, float(st["records"])], dtype=torch.float64, device="cuda")
    allstats = [torch.zeros_like(stats) for _ in range(world)]
    wall = torch.tensor([min(walls)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_gather(allstats, stats)
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
    else:
        allstats = [stats]
    out = None
    if rank == 0:
        per = [[float(x) for x in s.cpu()] for s in allstats]
        w = float(wall.cpu()[0])
        out = {"workload": "BASELINE.json configs[3] in shape: 24 contigs proportional to the human chromosomes, N runs, "
                           "soft-masked lower case; %.3f of the 3.1 Gbp genome (n_gpus / 8); defaults.toml architecture, "
                           "random-init weights; contig sharding; mapped FASTA file -> TSV text in host memory" % scale,
               "value": bases / w / 1e6, "unit": "Mbp/s", "seconds": w, "bases": bases, "scale": scale,
               "records": int(sum(p[5] for p in per)), "file_bytes": int(raw.size),
               "tsv_bytes_total": sum(p[0] for p in per), "rows_total": sum(p[1] for p in per),
               "h2d_bytes_total": sum(p[3] for p in per), "rank_seconds": [p[2] for p in per],
               "rank_forward_seconds": [p[4] for p in per], "generate_seconds": t_gen,
               "rank0_gpu_seconds": st["gpu_ms"] / 1e3, "rank0_waits_ms": st["waits_ms"]}
    del raw
    barrier()
    if rank == 0:
        for q in (path, path + ".json"):
            try:
                os.unlink(q)
            except OSError:
                pass
    return out


def chunk_sharded(args, rank, world, local_rank, ctx, stream, flush):
    """BASELINE.json configs[2]: ONE record split by position ranges over the ranks (halo recompute, no
    max-merge exchange); label (1 B) + score (4 B) per base are gathered to rank 0 over NCCL, which runs
    MSS, gap fill and segment extraction for the whole record.  Strong scaling: `value` = record bases /
    max-over-ranks time of the whole step.  The process group exists already; returns the result dict on rank 0."""
    import ctypes
    import torch
    import torch.distributed as dist
    from deepgrp_b200 import _lib, sharding

    weights = make_weights(args)
    handle = weights.device_handle(ctx)
    L = args.bases
    d_codes = torch.from_numpy(synth_codes(L, [1, 0])).cuda()       # the same record on every rank
    ranges = sharding.split_positions(L, world)
    p0, p1 = ranges[rank]
    pad = max(b - a for a, b in ranges)
    d_lab = torch.zeros(pad, dtype=torch.uint8, device="cuda")
    d_sc = torch.zeros(pad, dtype=torch.float32, device="cuda")
    labs = [torch.empty(pad, dtype=torch.uint8, device="cuda") for _ in range(world)] if rank == 0 else None
    scs = [torch.empty(pad, dtype=torch.float32, device="cuda") for _ in range(world)] if rank == 0 else None
    full_lab = torch.empty(L, dtype=torch.uint8, device="cuda") if rank == 0 else None
    full_sc = torch.empty(L, dtype=torch.float32, device="cuda") if rank == 0 else None
    n_rows = ctypes.c_int64(0)
    lib = _lib.lib()
    stage = {"range_ms": [], "finish_ms": []}

    def step():
        with torch.cuda.stream(stream):
            flush.zero_()
        _lib.check(lib.dgrp_predict_range_dev(
            ctx.handle, handle, ctypes.c_void_p(d_codes.data_ptr()), 0, L, L, p0, p1, STEP, BATCH,
            _lib.COMPAT_REFERENCE, ctypes.c_void_p(d_lab.data_ptr()), ctypes.c_void_p(d_sc.data_ptr())))
        stage["range_ms"].append(ctx.timings()["total_ms"])
        with torch.cuda.stream(stream):
            if world > 1:
                dist.gather(d_lab, labs, dst=0)
                dist.gather(d_sc, scs, dst=0)
            if rank == 0:
                for r, (a, b) in enumerate(ranges):
                    full_lab[a:b] = (labs[r] if world > 1 else d_lab)[:b - a]
                    full_sc[a:b] = (scs[r] if world > 1 else d_sc)[:b - a]
        if rank == 0:
            _lib.check(lib.dgrp_finish_record_dev(
                ctx.handle, ctypes.c_void_p(full_lab.data_ptr()), ctypes.c_void_p(full_sc.data_ptr()), L,
                5, 1, MIN_MSS, XDROP, ctypes.byref(n_rows)))
            stage["finish_ms"].append(ctx.timings()["total_ms"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    stage["range_ms"].clear()
    stage["finish_ms"].clear()
    launches0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop()
    t = torch.tensor([elapsed_ms, float(np.mean(stage["range_ms"]))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, range_ms = (float(x) for x in t.cpu())
    if rank != 0:
        return None
    cfg = workload_config(args, L)
    cfg["workload"] = (workload_name(args) + ", random-init weights seed 0, ONE synthetic iid-ACGT record split "
                       "by position ranges over the ranks")
    cfg["sharding"] = ("position ranges with halo recompute; NCCL gather of label (u8) + score (f32) to rank 0, "
                       "which runs MSS + segments for the whole record")
    finish_ms = float(np.mean(stage["finish_ms"]))
    return {
        "metric": "bases classified/sec (Mbp/s), record resident in HBM (device-timed)",
        "value": L * args.steps / (elapsed_ms / 1e3) / 1e6,
        "unit": "Mbp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks,
        "gpu_launches": int(launches),
        "stages_ms": {"range_forward_score_max_over_ranks": range_ms, "finish_mss_segments_rank0": finish_ms,
                      "gather_and_rest": elapsed_ms / args.steps - range_ms - finish_ms},
        "gather_bytes_per_step": 5 * (L - (ranges[0][1] - ranges[0][0])) if world > 1 else 0,
        "rows_per_step": int(n_rows.value), "mss_rounds": ctx.get_int("mss_rounds"),
    }


def run_chunk(args, rank, world, local_rank):
    """`--shard chunk`: the chunk-sharded run alone, as its own JSON line."""
    import torch
    import torch.distributed as dist
    from deepgrp_b200 import _lib
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    line = chunk_sharded(args, rank, world, local_rank, ctx, stream, flush)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bases", type=int, default=CONFIG2_BASES)
    ap.add_argument("--vecsize", type=int, default=T_DEFAULT)
    ap.add_argument("--units", type=int, default=U_DEFAULT)
    ap.add_argument("--ref-bases", type=int, default=750_000,
                    help="bases per CPU-reference step (bounded sample: ~10 s on the 16 host cores of a B200 box)")
    ap.add_argument("--rnn", default="GRU", choices=["GRU", "LSTM"])
    ap.add_argument("--weight-scale", type=float, default=1.0,
                    help="multiply the random-init weights (4 = the confident-output set of SURVEY.md section 8d)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sections", default="x4,strong,config5b,genome",
                    help="extra measurements attached to the JSON line: x4 (the confident-output weight set), strong "
                         "(BASELINE.json configs[2], one chr1-sized record chunk-sharded over the ranks), config5b (configs[4]: "
                         "T = 512, U = 128 on the same record length, chunk-sharded), genome "
                         "(configs[3] in shape, n_gpus/8 of the 3.1 Gbp multi-FASTA, end to end); '' for none")
    ap.add_argument("--e2e-api", default="stream", choices=["stream", "oneshot"])
    ap.add_argument("--early-rows", type=int, default=1,
                    help="e2e leg: 1 = a long record's rows leave slab by slab while it is still being computed "
                         "(dgrp_fasta_stream, DESIGN.md section 7), 0 = after the record's last window")
    ap.add_argument("--early-slabs", type=int, default=0, help="position slabs of a long record (0 = library default)")
    ap.add_argument("--mss-chunk", type=int, default=0, help="scores per thread of the MSS scan (0 = automatic)")
    ap.add_argument("--early-ratio", type=int, default=0, help="slab size relative to the one before, per cent (0 = library default)")
    ap.add_argument("--strong-bases", type=int, default=248_000_000)
    ap.add_argument("--genome-scale", type=float, default=0.0, help="fraction of the 3.1 Gbp genome (0 = n_gpus / 8)")
    ap.add_argument("--no-numa-bind", dest="numa_bind", action="store_false",
                    help="do not restrict the rank to the CPUs local to its GPU")
    ap.add_argument("--shard", default="contig", choices=["contig", "chunk"],
                    help="contig (default): one record per rank, weak scaling; chunk: ONE record split by "
                         "position ranges over the ranks (BASELINE.json configs[2], strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last `value` step's labels and rows (rank 0) as .npy "
                         "files in DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.shard != "contig"):
        ap.error("--dump-outputs writes the outputs of the default run (--impl ours --shard contig)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if (args.vecsize, args.units, args.rnn) != (T_DEFAULT, U_DEFAULT, "GRU") or args.bases != CONFIG2_BASES:
        # a custom shape: the attached sections describe the default architecture's other configurations
        if args.sections == ap.get_default("sections"):
            args.sections = ""
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.shard == "chunk":
        run_chunk(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
