"""Multi-GPU sharding of the prediction path (SURVEY.md section 8e): one process per GPU, no collective on
the data path.

* **By contig**: every rank reads the FASTA, decodes it on its GPU and derives the same assignment
  (:func:`assign_records`: largest record first, to the least loaded rank); it computes only its own
  records.  Rank 0 gathers the per-record TSV pieces and writes them in record order.
* **By position range inside one record**: a rank owning ``[p0, p1)`` recomputes every window whose
  placed rows intersect its range (halo recompute, no max-merge exchange) and yields ``uint8`` labels and
  ``float32`` scores; the record's owner concatenates the ranges and runs MSS + segment extraction
  (the MSS state machine needs the whole record).

The only communication is the gather of results (``torch.distributed``; ``gloo`` on CPU tensors works,
which is how tests/test_sharding.py exercises the plumbing without a GPU).
"""
from __future__ import annotations

import ctypes
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np


def assign_records(lengths: Sequence[int], world: int) -> List[int]:
    """Owner rank of every record: records sorted by length (descending, stable) go one by one to the
    rank with the smallest load so far (lowest rank on ties).  Mirrors the C++ in ``dgrp_predict_fasta``."""
    order = sorted(range(len(lengths)), key=lambda i: -int(lengths[i]))
    load = [0] * max(1, world)
    owner = [0] * len(lengths)
    for i in order:
        best = min(range(len(load)), key=lambda r: (load[r], r))
        owner[i] = best
        load[best] += int(lengths[i])
    return owner


def split_positions(length: int, parts: int, align: int = 1) -> List[Tuple[int, int]]:
    """``parts`` contiguous position ranges covering ``[0, length)`` (boundaries multiples of ``align``)."""
    cuts = [0]
    for k in range(1, parts):
        c = (length * k // parts) // align * align
        cuts.append(max(cuts[-1], c))
    cuts.append(length)
    return [(cuts[i], cuts[i + 1]) for i in range(parts)]


def gather_ranges(local_labels: np.ndarray, local_scores: np.ndarray, ranges: Sequence[Tuple[int, int]],
                  rank: int, world: int, owner: int = 0, dist=None):
    """Concentrate the per-range (label, score) arrays of one record on ``owner``.  Returns
    ``(labels uint8[L], scores float32[L])`` on the owner and ``(None, None)`` elsewhere."""
    import torch
    if world == 1:
        return local_labels, local_scores
    if dist is None:
        import torch.distributed as dist   # noqa: PLC0415
    sizes = [b - a for a, b in ranges]
    pad = max(sizes)
    lab = torch.zeros(pad, dtype=torch.uint8)
    sc = torch.zeros(pad, dtype=torch.float32)
    lab[:sizes[rank]] = torch.from_numpy(np.ascontiguousarray(local_labels))
    sc[:sizes[rank]] = torch.from_numpy(np.ascontiguousarray(local_scores))
    if rank == owner:
        labs = [torch.zeros(pad, dtype=torch.uint8) for _ in range(world)]
        scs = [torch.zeros(pad, dtype=torch.float32) for _ in range(world)]
        dist.gather(lab, labs, dst=owner)
        dist.gather(sc, scs, dst=owner)
        labels = np.concatenate([labs[r][:sizes[r]].numpy() for r in range(world)])
        scores = np.concatenate([scs[r][:sizes[r]].numpy() for r in range(world)])
        return labels, scores
    dist.gather(lab, None, dst=owner)
    dist.gather(sc, None, dst=owner)
    return None, None


def predict_range(model, codes: np.ndarray, length: int, p0: int, p1: int, step_size: int,
                  batch_size: int, compat: int = 0, codes_base: int = 0):
    """(labels uint8, scores float32) of positions ``[p0, p1)`` of a record (``dgrp_predict_range``)."""
    from . import _lib
    ctx = _lib.context()
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    lab = np.zeros(p1 - p0, np.uint8)
    sc = np.zeros(p1 - p0, np.float32)
    _lib.check(_lib.lib().dgrp_predict_range(
        ctx.handle, model.device_handle(ctx), _lib.ptr(codes), codes_base, codes.size, length, p0, p1,
        int(step_size), int(batch_size), compat, _lib.ptr(lab), _lib.ptr(sc)))
    return lab, sc


def finish_record(labels: np.ndarray, scores: np.ndarray, n_classes: int, use_mss: bool,
                  min_mss_len: int, xdrop_len: int, startpos: int):
    """MSS gap fill + segment rows from gathered (label, score) of a whole record
    (``dgrp_finish_record``): returns (labels uint8[L], rows).  ``use_mss`` must be true: without MSS the
    reference's labels are the argmax after a softmax over the whole record's maximum, which can round two close
    probabilities into a tie that the ranges' labels (argmax of the raw vote) do not reproduce."""
    if not use_mss:
        raise ValueError("finish_record needs use_mss: without MSS the labels depend on the whole record's "
                         "softmax, which the ranges' labels do not carry; predict the record whole")
    from . import _lib
    ctx = _lib.context()
    labels = np.ascontiguousarray(labels, dtype=np.uint8)
    scores = np.ascontiguousarray(scores, dtype=np.float32)
    out = np.zeros_like(labels)
    cap = 4096
    while True:
        rows = np.zeros(cap, dtype=_lib.ROW_DTYPE)
        n_rows = ctypes.c_int64(0)
        rc = _lib.lib().dgrp_finish_record(ctx.handle, _lib.ptr(labels), _lib.ptr(scores), labels.size,
                                           n_classes, int(use_mss), int(min_mss_len), int(xdrop_len),
                                           int(startpos), _lib.ptr(out), _lib.ptr(rows), cap,
                                           ctypes.byref(n_rows))
        if rc == _lib.E_CAPACITY:
            cap = int(n_rows.value)
            continue
        _lib.check(rc)
        return out, rows[:n_rows.value]


def predict_record_sharded(compute_range: Callable[[int, int], Tuple[np.ndarray, np.ndarray]],
                           finish: Callable[[np.ndarray, np.ndarray], object], length: int, rank: int,
                           world: int, owner: int = 0, dist=None):
    """One record split by position across ``world`` ranks: ``compute_range(p0, p1)`` runs on every rank
    for its own range, the owner gathers and calls ``finish(labels, scores)``."""
    ranges = split_positions(length, world)
    p0, p1 = ranges[rank]
    lab, sc = compute_range(p0, p1)
    labels, scores = gather_ranges(lab, sc, ranges, rank, world, owner, dist)
    if rank == owner:
        return finish(labels, scores)
    return None


def merge_record_texts(pieces: Sequence[Sequence[Tuple[int, bytes]]]) -> bytes:
    """Rank 0: per-rank lists of (record index, TSV bytes) -> the file's TSV in record order."""
    allp = sorted((p for rank_list in pieces for p in rank_list), key=lambda t: t[0])
    return b"".join(t[1] for t in allp)


def stream_slabs(length: int, vecsize: int, step_size: int, unit_windows: int = 0, n_slabs: int = 0,
                 ratio_pct: int = 0) -> np.ndarray:
    """The position slabs ``dgrp_fasta_stream_*`` cuts a long record into for its early rows (C ABI
    ``dgrp_fasta_stream_plan``; host arithmetic, no GPU needed): the slab ends, the last one ``length``; empty when
    the record is too short for that route."""
    import ctypes
    from . import _lib
    ends = np.zeros(64, np.int64)
    n = ctypes.c_int(0)
    _lib.check(_lib.lib().dgrp_fasta_stream_plan(int(length), int(vecsize), int(step_size), int(unit_windows),
                                                 int(n_slabs), int(ratio_pct), _lib.ptr(ends), 64, ctypes.byref(n)))
    return ends[:n.value].copy()


def fasta_slices(raw, world: int = 1):
    """The host index of the streaming driver (C ABI ``dgrp_fasta_index``; no GPU needed): ``(cuts, owner)`` --
    ``cuts[k]:cuts[k+1]`` is slice ``k`` of the FASTA text (whole records, >= 8 MiB unless the file ends) and
    ``owner[k]`` the rank it goes to, largest slice first to the least loaded rank."""
    import ctypes
    from . import _lib
    n = len(raw)
    buf = np.frombuffer(raw, dtype=np.uint8) if n else np.zeros(0, np.uint8)
    cap = max(1, n // (8 << 20) + 2)
    cuts, owner = np.zeros(cap + 1, np.int64), np.zeros(cap, np.int32)
    ns = ctypes.c_int64(0)
    _lib.check(_lib.lib().dgrp_fasta_index(_lib.ptr(buf), n, int(world), _lib.ptr(cuts), _lib.ptr(owner), cap,
                                           ctypes.byref(ns)))
    return cuts[:ns.value + 1].copy(), owner[:ns.value].copy()
