"""deepgrp_b200.prediction -- drop-in for the reference's ``deepgrp.prediction`` on the prediction
path (``deepgrp/prediction.py:14-141``): same function names and argument meaning.

Differences that callers can see:

* ``fetch_validation_batch`` returns a :class:`WindowDataset` (a lazy window descriptor that can be
  iterated batch by batch exactly like the reference's ``tf.data.Dataset``) instead of a TensorFlow
  dataset.  When it is handed to :func:`predict` together with a :class:`~deepgrp_b200.model.ModelWeights`
  the windows are never materialised: the one-hot matrix is turned into base codes on the GPU and
  the fused kernel reads windows as strided views (``csrc/forward.cu``).
* ``predict`` reproduces the reference's placement of the final short batch
  (``deepgrp/prediction.py:105``, SURVEY.md section 0 fact 3) by default; ``compat="fixed"`` places
  every window at ``w * step``.
"""
from __future__ import annotations

import ctypes
import io
import os
from typing import Iterator, Optional, Tuple

import numpy as np

from . import _lib
from . import mss
from . import sequence as dgsequence
from .model import ModelWeights, Options, create_model, load_model
from . import preprocessing  # noqa: F401  (Data, as in the reference's import list)

_COMPAT = {"reference": _lib.COMPAT_REFERENCE, "fixed": _lib.COMPAT_FIXED}
_MASK = {"soft": _lib.MASK_SOFT, "hard": _lib.MASK_HARD}
TRACK_BIN_MAX = 1_000_000


class WindowDataset:
    """Windows ``data.T[i:i+vecsize]`` for ``i in range(0, L - vecsize, step_size)`` in batches of
    ``batch_size`` (the final batch may be short), reference ``deepgrp/prediction.py:28-37``."""

    def __init__(self, data: np.ndarray, step_size: int, batch_size: int, vecsize: int):
        self.data = np.asarray(data)
        self.step_size = int(step_size)
        self.batch_size = int(batch_size)
        self.vecsize = int(vecsize)

    @property
    def length(self) -> int:
        return int(self.data.shape[1])

    def window_starts(self) -> range:
        return range(0, self.length - self.vecsize, self.step_size)     # end EXCLUSIVE

    def __len__(self) -> int:
        n = len(self.window_starts())
        return (n + self.batch_size - 1) // self.batch_size

    def __iter__(self) -> Iterator[np.ndarray]:
        data_t = self.data.T
        starts = self.window_starts()
        for b in range(0, len(starts), self.batch_size):
            idx = starts[b:b + self.batch_size]
            yield np.stack([data_t[i:i + self.vecsize].astype("float32") for i in idx])


def fetch_validation_batch(data: np.ndarray, step_size: int, batch_size: int,
                           vecsize: int) -> WindowDataset:
    """Reference ``deepgrp/prediction.py:14-37`` (no randomisation)."""
    return WindowDataset(data, step_size, batch_size, vecsize)


def forward_windows(model: ModelWeights, batch) -> np.ndarray:
    """``keras.Model.predict_on_batch``: ``float32[B, T, 5]`` windows -> ``float32[B, T, C]``."""
    batch = np.ascontiguousarray(batch, dtype=np.float32)
    if batch.ndim != 3 or batch.shape[1] != model.vecsize or batch.shape[2] != 5:
        raise ValueError("expected windows of shape [B, %d, 5], got %s" % (model.vecsize, batch.shape))
    ctx = _lib.context()
    out = np.zeros((batch.shape[0], model.vecsize, model.n_classes), dtype=np.float32)
    _lib.check(_lib.lib().dgrp_forward_windows(ctx.handle, model.device_handle(ctx), _lib.ptr(batch),
                                               batch.shape[0], _lib.ptr(out)))
    return out


def apply_mss(probs: np.ndarray, options: Options) -> np.ndarray:
    """argmax + logit score -> maximal scoring segments -> gap-filled one-hot ``float64[n, C]``
    (reference ``deepgrp/prediction.py:40-59``)."""
    probs = np.ascontiguousarray(probs, dtype=np.float32)
    n, nof = probs.shape
    out = np.zeros((n, nof), dtype=np.float64)
    if n == 0:
        return out
    ctx = _lib.context()
    _lib.check(_lib.lib().dgrp_apply_mss(ctx.handle, _lib.ptr(probs), n, nof,
                                         int(options.min_mss_len), int(options.xdrop_len),
                                         _lib.ptr(out)))
    return out


def mss_scores(probs: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """The score transform of ``apply_mss`` alone (reference ``deepgrp/prediction.py:51-57``):
    ``(float64 scores, int64 classes)``."""
    probs = np.ascontiguousarray(probs, dtype=np.float32)
    n, nof = probs.shape
    scores = np.zeros(n, dtype=np.float64)
    classes = np.zeros(n, dtype=np.int64)
    if n:
        ctx = _lib.context()
        _lib.check(_lib.lib().dgrp_mss_scores(ctx.handle, _lib.ptr(probs), n, nof, _lib.ptr(scores),
                                              _lib.ptr(classes)))
    return scores, classes


def softmax(array: np.ndarray) -> np.ndarray:
    """``exp(x - max(x)) / rowsum`` (reference ``deepgrp/prediction.py:62-65``)."""
    array = np.ascontiguousarray(array, dtype=np.float32)
    out = np.zeros_like(array)
    if array.size:
        ctx = _lib.context()
        _lib.check(_lib.lib().dgrp_softmax(ctx.handle, _lib.ptr(array), array.shape[0],
                                           array.shape[1], _lib.ptr(out)))
    return out


def setup_prediction_from_options_checkpoint(options: Options, logdir) -> ModelWeights:
    """Reference ``deepgrp/prediction.py:68-86``: the model of ``options`` with the weights of the latest
    checkpoint in ``logdir``.  ``logdir`` may hold TensorFlow-format checkpoints as the reference's
    training writes them (``ModelCheckpoint(save_weights_only=True)``, ``deepgrp/training.py:53-59``; read
    by :mod:`deepgrp_b200.tfckpt` without TensorFlow), or a Keras ``.hdf5`` / ``.h5`` / ``.npz`` weights file
    (the newest wins); it may also be such a file itself."""
    path = os.fspath(logdir)
    if os.path.isdir(path):
        from . import tfckpt
        prefix = tfckpt.latest_checkpoint(path)
        if prefix is not None:
            w = tfckpt.deepgrp_weights(tfckpt.read_bundle(prefix))
            return ModelWeights(int(options.vecsize), int(w["recurrent_kernel"].shape[0]), w["kernel"],
                                w["recurrent_kernel"], w["bias"], w["ff_kernel"], w["ff_bias"],
                                w.get("att_scale"), w["rnn"])
        cands = [os.path.join(path, f) for f in os.listdir(path)
                 if f.endswith((".hdf5", ".h5", ".npz"))]
        if not cands:
            raise FileNotFoundError("no TensorFlow checkpoint and no .hdf5/.h5/.npz weights in %s" % path)
        path = max(cands, key=os.path.getmtime)
    model = load_model(path)
    if model.vecsize != options.vecsize:
        model.vecsize = int(options.vecsize)     # weights do not depend on the window length
    return model


def predict(model, data, results_shape: Tuple[int, int], step_size: int,
            compat: str = "reference") -> np.ndarray:
    """Predict for a complete sequence (reference ``deepgrp/prediction.py:89-111``): every window's
    class probabilities are merged into ``float32[L, C]`` by elementwise maximum."""
    # The fused route enumerates AND places windows with one step, so it only applies when the dataset was
    # built with the step `predict` is called with (the reference enumerates with the dataset's step and places
    # with predict's), on an integer one-hot matrix; anything else takes the reference's literal loop below.
    if isinstance(model, ModelWeights) and isinstance(data, WindowDataset) \
            and data.vecsize == model.vecsize and data.data.shape[0] == 5 \
            and tuple(results_shape) == (data.length, model.n_classes) \
            and int(step_size) == step_size and data.step_size == int(step_size) \
            and np.issubdtype(np.asarray(data.data).dtype, np.integer):
        fwd = np.ascontiguousarray(data.data, dtype=np.int8)
        predictions = np.zeros(results_shape, dtype=np.float32)
        if data.length:
            ctx = _lib.context()
            _lib.check(_lib.lib().dgrp_predict_onehot(
                ctx.handle, model.device_handle(ctx), _lib.ptr(fwd), data.length, int(step_size),
                data.batch_size, _COMPAT[compat], _lib.ptr(predictions)))
        return predictions
    # generic route, literally the reference loop: any object with predict_on_batch, any iterable
    predictions = np.zeros(results_shape, dtype=np.float32)
    for i, batch in enumerate(data):
        index = i * batch.shape[0] * step_size
        probas = np.ascontiguousarray(model.predict_on_batch(batch), dtype=np.float32)
        dgsequence.get_max(predictions[index:], probas, step_size)
    return predictions


def predict_complete(step_size: int, options: Options, logdir, data, use_mss: bool = False
                     ) -> np.ndarray:
    """Restores a model and predicts for a sequence (reference ``deepgrp/prediction.py:114-141``)."""
    model = setup_prediction_from_options_checkpoint(options, logdir)
    val_iterator = fetch_validation_batch(data.fwd, step_size, options.batch_size, options.vecsize)
    output_shape = data.truelbl.shape[::-1]
    predictions = predict(model, val_iterator, output_shape, step_size)
    if use_mss:
        return apply_mss(predictions, options)
    return softmax(predictions)


def predict_sequence(model: ModelWeights, raw: bytes, step_size: int, batch_size: int,
                     use_mss: bool, min_mss_len: int, xdrop_len: int, fold_case: bool = True,
                     compat: str = "reference", want_labels: bool = True):
    """One record end to end on the GPU (the body of ``_predict`` + ``yield_segments``, reference
    ``deepgrp/__main__.py:46-83, 288-290``): raw sequence bytes -> (labels uint8[L], startpos, rows).
    ``rows`` is a structured array (start, end, label, record) of the label > 0 segments."""
    ctx = _lib.context()
    n = len(raw)
    buf = np.frombuffer(raw, dtype=np.uint8) if n else np.zeros(0, np.uint8)
    labels = np.zeros(n, dtype=np.uint8) if want_labels else None
    cap = 4096
    while True:
        rows = np.zeros(cap, dtype=_lib.ROW_DTYPE)
        start, length, n_rows = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
        rc = _lib.lib().dgrp_predict_sequence(
            ctx.handle, model.device_handle(ctx), _lib.ptr(buf), n, int(fold_case), int(step_size),
            int(batch_size), int(use_mss), int(min_mss_len), int(xdrop_len), _COMPAT[compat],
            ctypes.byref(start), ctypes.byref(length), _lib.ptr(labels), _lib.ptr(rows), cap,
            ctypes.byref(n_rows))
        if rc == _lib.E_CAPACITY:
            cap = int(n_rows.value)
            continue
        if rc == _lib.E_ALLN:
            raise ValueError("negative dimensions are not allowed")
        _lib.check(rc)
        break
    if labels is not None:
        labels = labels[:length.value]
    return labels, int(start.value), rows[:n_rows.value]


def predict_fasta(model: ModelWeights, raw: bytes, step_size: int, batch_size: int, use_mss: bool,
                  min_mss_len: int, xdrop_len: int, compat: str = "reference"):
    """A whole (multi-)FASTA file in one call: raw file bytes -> (rows, records).  The text is decoded
    on the GPU (reference ``deepgrp/__main__.py:20-43``) and every record runs the fused device
    pipeline.  ``rows``: structured array (start, end, label, record); ``records``: list of
    ``(header, startpos, length)``.  A blank line raises ``IndexError`` and an all-'N' record
    ``ValueError``, as the reference does."""
    n_rows, records = _predict_fasta_call(model, raw, step_size, batch_size, use_mss, min_mss_len, xdrop_len,
                                          compat)
    rows = np.zeros(n_rows, dtype=_lib.ROW_DTYPE)
    if n_rows:
        _lib.check(_lib.lib().dgrp_fasta_rows(_lib.context().handle, _lib.ptr(rows), n_rows))
    return rows, records


def _predict_fasta_call(model: ModelWeights, raw, step_size: int, batch_size: int, use_mss: bool,
                        min_mss_len: int, xdrop_len: int, compat: str):
    """``dgrp_predict_fasta`` -> (number of rows, records); the rows stay in the context."""
    ctx = _lib.context()
    n = len(raw)
    buf = np.frombuffer(raw, dtype=np.uint8) if n else np.zeros(0, np.uint8)
    n_rows, n_rec = ctypes.c_int64(0), ctypes.c_int64(0)
    rc = _lib.lib().dgrp_predict_fasta(
        ctx.handle, model.device_handle(ctx), _lib.ptr(buf), n, int(step_size), int(batch_size),
        int(use_mss), int(min_mss_len), int(xdrop_len), _COMPAT[compat], ctypes.byref(n_rows),
        ctypes.byref(n_rec))
    if rc == _lib.E_FASTA:
        raise IndexError("string index out of range")
    if rc == _lib.E_ALLN:
        raise ValueError("negative dimensions are not allowed")
    _lib.check(rc)
    k = n_rec.value
    off, ln = np.zeros(k, np.int64), np.zeros(k, np.int64)
    sp, le = np.zeros(k, np.int64), np.zeros(k, np.int64)
    if k:
        _lib.check(_lib.lib().dgrp_fasta_records(ctx.handle, _lib.ptr(off), _lib.ptr(ln),
                                                 _lib.ptr(sp), _lib.ptr(le), k))
    records = [(bytes(raw[off[i]:off[i] + ln[i]]).decode("utf-8", "replace"), int(sp[i]), int(le[i]))
               for i in range(k)]
    return int(n_rows.value), records


def _fasta_tsv_call(model: ModelWeights, raw, filename: str, step_size: int, batch_size: int,
                    use_mss: bool, min_mss_len: int, xdrop_len: int, compat: str):
    """-> (memoryview of the TSV text, number of rows, number of records)."""
    ctx = _lib.context()
    n = len(raw)
    buf = np.frombuffer(raw, dtype=np.uint8) if n else np.zeros(0, np.uint8)
    tsv, tsv_len = ctypes.c_void_p(), ctypes.c_int64(0)
    n_rows, n_rec = ctypes.c_int64(0), ctypes.c_int64(0)
    rc = _lib.lib().dgrp_predict_fasta_tsv(
        ctx.handle, model.device_handle(ctx), _lib.ptr(buf), n, os.fsencode(filename),
        int(step_size), int(batch_size), int(use_mss), int(min_mss_len), int(xdrop_len),
        _COMPAT[compat], ctypes.byref(tsv), ctypes.byref(tsv_len), ctypes.byref(n_rows),
        ctypes.byref(n_rec))
    if rc == _lib.E_FASTA:
        raise IndexError("string index out of range")
    if rc == _lib.E_ALLN:
        raise ValueError("negative dimensions are not allowed")
    _lib.check(rc)
    if tsv_len.value == 0:
        return memoryview(b""), int(n_rows.value), int(n_rec.value)
    view = memoryview((ctypes.c_ubyte * tsv_len.value).from_address(tsv.value)).cast("B").toreadonly()
    return view, int(n_rows.value), int(n_rec.value)


def predict_fasta_tsv_view(model: ModelWeights, raw, filename: str, step_size: int,
                           batch_size: int, use_mss: bool, min_mss_len: int, xdrop_len: int,
                           compat: str = "reference") -> memoryview:
    """The TSV text ``deepgrp predict`` writes for one file (reference ``deepgrp/__main__.py:288-292``),
    formatted on the GPU.  Returns a read-only view of pinned host memory owned by the context: it is
    valid until the next prediction call, so write it out (or copy it) first."""
    return _fasta_tsv_call(model, raw, filename, step_size, batch_size, use_mss, min_mss_len,
                           xdrop_len, compat)[0]


class FastaTsvStream:
    """Pipelined whole-file prediction (C ABI ``dgrp_fasta_stream_*``; reference ``deepgrp/__main__.py:275-295``
    writes a record's rows as soon as the record is done).  Iterating yields ``(slice, ordinal, n_rows, last,
    view)`` per piece of TSV text, in file order of this rank's records; ``view`` is a read-only memoryview of
    pinned host memory that is valid until the next iteration -- write it out or copy it.  A blank line
    (``IndexError``) or an all-``N`` record (``ValueError``) is raised after the text of the records before it.
    ``raw`` must stay alive while the stream is open (a reference is kept)."""

    def __init__(self, model: ModelWeights, raw, filename: str, step_size: int, batch_size: int, use_mss: bool,
                 min_mss_len: int, xdrop_len: int, compat: str = "reference", rank: int = 0, world: int = 1):
        self._ctx = _lib.context()
        self._raw = raw
        n = len(raw)
        self._buf = np.frombuffer(raw, dtype=np.uint8) if n else np.zeros(0, np.uint8)
        self._handle = ctypes.c_void_p()
        self._ctx.set_int("shard_rank", rank)
        self._ctx.set_int("shard_world", world)
        try:
            _lib.check(_lib.lib().dgrp_fasta_stream_open(
                self._ctx.handle, model.device_handle(self._ctx), _lib.ptr(self._buf), n, os.fsencode(filename),
                int(step_size), int(batch_size), int(use_mss), int(min_mss_len), int(xdrop_len), _COMPAT[compat],
                ctypes.byref(self._handle)))
        finally:
            self._ctx.set_int("shard_rank", 0)
            self._ctx.set_int("shard_world", 1)

    def __iter__(self):
        return self

    def __next__(self):
        if not self._handle:
            raise StopIteration
        tsv, tsv_len = ctypes.c_void_p(), ctypes.c_int64(0)
        sl, od, nr = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
        last, done = ctypes.c_int(0), ctypes.c_int(0)
        rc = _lib.lib().dgrp_fasta_stream_next(self._handle, ctypes.byref(tsv), ctypes.byref(tsv_len),
                                               ctypes.byref(sl), ctypes.byref(od), ctypes.byref(nr),
                                               ctypes.byref(last), ctypes.byref(done))
        if rc != 0 or done.value:
            self.stats = self._stats()
            self.close()
            if rc == _lib.E_FASTA:
                raise IndexError("string index out of range")
            if rc == _lib.E_ALLN:
                raise ValueError("negative dimensions are not allowed")
            _lib.check(rc)
            raise StopIteration
        if tsv_len.value == 0:
            view = memoryview(b"")
        else:
            view = memoryview((ctypes.c_ubyte * tsv_len.value).from_address(tsv.value)).cast("B").toreadonly()
        return int(sl.value), int(od.value), int(nr.value), bool(last.value), view

    def _stats(self) -> dict:
        v = [ctypes.c_int64(0) for _ in range(7)]
        f, g = ctypes.c_double(0.0), ctypes.c_double(0.0)
        _lib.check(_lib.lib().dgrp_fasta_stream_stats(self._handle, *[ctypes.byref(x) for x in v],
                                                      ctypes.byref(f), ctypes.byref(g)))
        names = ("rows", "records", "bases", "windows", "launches", "h2d_bytes", "d2h_bytes")
        out = {k: int(x.value) for k, x in zip(names, v)}
        out["forward_ms"], out["gpu_ms"] = float(f.value), float(g.value)
        w = (ctypes.c_double * 12)()
        _lib.check(_lib.lib().dgrp_fasta_stream_waits(self._handle, w))
        out["waits_ms"] = dict(zip(("compute_for_upload", "compute_for_text_buffer", "copier_for_record",
                                    "copier_for_slot", "copier_copies", "uploader_for_buffer", "uploader_copying",
                                    "compute_total", "decode", "records_host", "tsv", "encode"),
                                   (float(x) for x in w)))
        return out

    def close(self) -> None:
        if self._handle:
            _lib.lib().dgrp_fasta_stream_close(self._handle)
            self._handle = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:       # interpreter shutdown
            pass


def predict_fasta_tsv_stream(model: ModelWeights, raw, filename: str, outstream, step_size: int, batch_size: int,
                             use_mss: bool, min_mss_len: int, xdrop_len: int, compat: str = "reference",
                             rank: int = 0, world: int = 1) -> dict:
    """Write the TSV text of ``raw`` (one FASTA file) to the binary stream ``outstream`` piece by piece as the
    records finish; returns the stream's totals (rows, records, bases, ...)."""
    with FastaTsvStream(model, raw, filename, step_size, batch_size, use_mss, min_mss_len, xdrop_len, compat,
                        rank, world) as st:
        for _, _, _, _, view in st:
            if len(view):
                outstream.write(view)
        return st.stats


def predict_fasta_tsv_sharded(model: ModelWeights, raw, filename: str, step_size: int, batch_size: int,
                              use_mss: bool, min_mss_len: int, xdrop_len: int, rank: int, world: int,
                              compat: str = "reference"):
    """Contig-sharded form of :func:`predict_fasta_tsv_view`: this rank computes only the records the
    largest-first assignment gives it and returns ``[(record index, TSV bytes), ...]`` for them; merge
    the per-rank lists with :func:`deepgrp_b200.sharding.merge_record_texts`."""
    ctx = _lib.context()
    ctx.set_int("shard_rank", rank)
    ctx.set_int("shard_world", world)
    try:
        view, _, n_rec = _fasta_tsv_call(model, raw, filename, step_size, batch_size, use_mss,
                                         min_mss_len, xdrop_len, compat)
        owner, off, ln = (np.zeros(max(n_rec, 1), np.int64) for _ in range(3))
        if n_rec:
            _lib.check(_lib.lib().dgrp_fasta_record_tsv(ctx.handle, _lib.ptr(owner), _lib.ptr(off),
                                                        _lib.ptr(ln), n_rec))
        return [(k, bytes(view[off[k]:off[k] + ln[k]])) for k in range(n_rec)
                if owner[k] == rank and ln[k] > 0]
    finally:
        ctx.set_int("shard_rank", 0)
        ctx.set_int("shard_world", 1)


def predict_fasta_tsv(model: ModelWeights, raw, filename: str, step_size: int, batch_size: int,
                      use_mss: bool, min_mss_len: int, xdrop_len: int,
                      compat: str = "reference") -> str:
    """``predict_fasta_tsv_view`` copied into a ``str``."""
    return bytes(predict_fasta_tsv_view(model, raw, filename, step_size, batch_size, use_mss,
                                        min_mss_len, xdrop_len, compat)).decode("utf-8", "replace")


def _mask_mode(mode: str) -> int:
    if mode not in _MASK:
        raise ValueError("mask mode must be 'soft' or 'hard', not %r" % (mode,))
    return _MASK[mode]


def mask_fasta(raw, rows: np.ndarray, mode: str = "soft") -> bytes:
    """The FASTA text ``raw`` with the positions that ``rows`` cover masked, on the GPU: lower-cased (``soft``,
    ASCII ``A``-``Z`` only) or replaced by ``N`` (``hard``).  ``rows`` is the structured array
    :func:`predict_fasta` returns (``record`` indexes the records with a non-empty header, untrimmed
    coordinates); it must be sorted by (record, start) and disjoint within a record.  Every other byte is copied
    unchanged, so the result has the length of ``raw``.  A blank line raises ``IndexError``."""
    code = _mask_mode(mode)
    ctx = _lib.context()
    n = len(raw)
    buf = np.frombuffer(raw, dtype=np.uint8) if n else np.zeros(0, np.uint8)
    rows = np.ascontiguousarray(rows, dtype=_lib.ROW_DTYPE)
    out = np.empty(max(n, 1), dtype=np.uint8)
    rc = _lib.lib().dgrp_mask_fasta(ctx.handle, _lib.ptr(buf), n, _lib.ptr(rows), rows.size, code, _lib.ptr(out))
    if rc == _lib.E_FASTA:
        raise IndexError("string index out of range")
    _lib.check(rc)
    return out[:n].tobytes()


def predict_fasta_tsv_masked(model: ModelWeights, raw, filename: str, outstream, maskstream, step_size: int,
                             batch_size: int, use_mss: bool, min_mss_len: int, xdrop_len: int, mode: str = "soft",
                             compat: str = "reference") -> dict:
    """:func:`predict_fasta_tsv_stream` that also writes the masked text of ``raw`` (see :func:`mask_fasta`) to
    the binary stream ``maskstream``: :func:`predict_fasta_sliced` with a mask stream."""
    return predict_fasta_sliced(model, raw, filename, outstream, step_size, batch_size, use_mss, min_mss_len,
                                xdrop_len, compat, maskstream=maskstream, mask_mode=mode)


def _track_bin(bin: int) -> int:
    if int(bin) != bin or not 1 <= bin <= TRACK_BIN_MAX:
        raise ValueError("track bin size must be an integer in [1, %d], not %r" % (TRACK_BIN_MAX, bin))
    return int(bin)


def track_last(cls: int, bin: int) -> memoryview:
    """``dgrp_track_last``: the bedGraph text of class ``cls`` of the last :func:`predict_fasta` call, which ran with
    the context option ``keep_votes`` set.  A read-only view of pinned host memory owned by the context, valid until
    the next call: write it out (or copy it) first."""
    ctx = _lib.context()
    text, n = ctypes.c_void_p(), ctypes.c_int64(0)
    _lib.check(_lib.lib().dgrp_track_last(ctx.handle, int(cls), int(bin), ctypes.byref(text), ctypes.byref(n)))
    if n.value == 0:
        return memoryview(b"")
    return memoryview((ctypes.c_ubyte * n.value).from_address(text.value)).cast("B").toreadonly()


def predict_fasta_sliced(model: ModelWeights, raw, filename: str, outstream, step_size: int, batch_size: int,
                         use_mss: bool, min_mss_len: int, xdrop_len: int, compat: str = "reference", maskstream=None,
                         mask_mode: str = "soft", trackstreams: Optional[dict] = None, track_bin: int = 10) -> dict:
    """Predict one FASTA file slice by slice (whole records, >= 8 MiB, the streaming driver's cuts with one rank),
    which bounds device memory.  One prediction per slice serves every output:

    * ``outstream`` (binary, or None): the TSV text, as :func:`predict_fasta_tsv_stream` writes it;
    * ``maskstream`` (binary, or None): the masked text of the slice (see :func:`mask_fasta`, ``mask_mode``), made
      from its rows while they are still on the device;
    * ``trackstreams`` (``{class: binary stream}``, or None): the bedGraph lines of each class with bins of
      ``track_bin`` bases (see :func:`predict_fasta_tracks`), from the slice's max-vote rows kept on the device.

    A slice with a blank line or an all-``N`` record is run again through :func:`predict_fasta_tsv_stream` (when there
    is an ``outstream``), so the TSV text holds the rows of the records before the error, as the default route writes
    them, and the same ``IndexError`` / ``ValueError`` is raised; the masked text and the tracks then hold the slices
    before that one.  Returns the totals (rows, records, bases, slices)."""
    from .sharding import fasta_slices
    code = _mask_mode(mask_mode) if maskstream is not None else None
    if trackstreams:
        track_bin = _track_bin(track_bin)
        bad = [c for c in trackstreams if not 1 <= int(c) < model.n_classes]
        if bad:
            raise ValueError("track classes must lie in [1, %d), got %s" % (model.n_classes, bad))
    ctx = _lib.context()
    cuts, _ = fasta_slices(raw, 1)
    whole = memoryview(raw) if len(raw) else memoryview(b"")
    totals = {"rows": 0, "records": 0, "bases": 0, "slices": len(cuts) - 1}
    for k in range(len(cuts) - 1):
        piece = whole[int(cuts[k]):int(cuts[k + 1])]
        keep = ctx.get_int("keep_votes")          # the caller's setting, restored after the call
        if trackstreams:
            ctx.set_int("keep_votes", 1)
        try:
            if outstream is not None:
                view, n_rows, n_rec = _fasta_tsv_call(model, piece, filename, step_size, batch_size, use_mss,
                                                      min_mss_len, xdrop_len, compat)
            else:
                n_rows, recs = _predict_fasta_call(model, piece, step_size, batch_size, use_mss, min_mss_len,
                                                   xdrop_len, compat)
                view, n_rec = memoryview(b""), len(recs)
        except (IndexError, ValueError):
            if outstream is None:
                raise
            predict_fasta_tsv_stream(model, piece, filename, outstream, step_size, batch_size, use_mss,
                                     min_mss_len, xdrop_len, compat)
            raise RuntimeError("slice %d failed in the whole-slice call but not in the stream" % k)
        finally:
            ctx.set_int("keep_votes", keep)
        totals["bases"] += int(ctx.timings()["bases"])
        totals["rows"] += n_rows
        totals["records"] += n_rec
        if len(view):
            outstream.write(view)
        n = len(piece)
        if maskstream is not None and n:
            buf = np.frombuffer(piece, dtype=np.uint8)
            out = np.empty(n, dtype=np.uint8)
            _lib.check(_lib.lib().dgrp_mask_fasta_last(ctx.handle, _lib.ptr(buf), n, code, _lib.ptr(out)))
            maskstream.write(out)
        for cls, stream in (trackstreams or {}).items():
            text = track_last(cls, track_bin)
            if len(text):
                stream.write(text)
    return totals


def predict_fasta_tracks(model: ModelWeights, raw, step_size: int, batch_size: int, bin: int = 10,
                         compat: str = "reference") -> dict:
    """Per-base repeat probability tracks of one FASTA file: ``{class: bedGraph bytes}`` for every repeat class
    ``1 .. C-1``, computed and formatted on the GPU.  The value of a position is its max-vote probability
    (:func:`predict`, before MSS or softmax) in untrimmed record coordinates; positions outside a record's span
    ``[startpos, startpos + length)`` (its edge ``N`` s) have none.  Bins ``[k bin, (k + 1) bin)`` are aligned to 0 and
    clipped to the span; a bin's value is ``rint(mean * 1000) / 1000`` (float64 sum in position order, round half to
    even), written as ``%d.%03d``.  Consecutive bins of one record with the same value make one line
    ``chrom\tstart\tend\tvalue``; ``chrom`` is the header's first word.  The file runs in slices (whole records,
    >= 8 MiB).  A blank line raises ``IndexError`` and an all-``N`` record ``ValueError``, as in ``predict``."""
    bin = _track_bin(bin)
    streams = {c: io.BytesIO() for c in range(1, model.n_classes)}
    predict_fasta_sliced(model, raw, "", None, step_size, batch_size, False, 50, 50, compat,
                         trackstreams=streams, track_bin=bin)
    return {c: s.getvalue() for c, s in streams.items()}


# ---- evaluation helpers (deepgrp/prediction.py:144-260; used by deepgrp/optimization.py:58-69) -------

def calculate_multiclass_matthews_cc(cnf_matrix: np.ndarray) -> float:
    """R_K / multi-class Matthews correlation coefficient of a confusion matrix
    (deepgrp/prediction.py:144-164; O(C^2) host arithmetic on the GPU-built matrix)."""
    t_sum = cnf_matrix.sum(axis=1, dtype=float)
    p_sum = cnf_matrix.sum(axis=0, dtype=float)
    n_correct = np.trace(cnf_matrix, dtype=float)
    n_samples = p_sum.sum()
    cov_ytyp = n_correct * n_samples - np.dot(t_sum, p_sum)
    cov_ypyp = n_samples**2 - np.dot(p_sum, p_sum)
    cov_ytyt = n_samples**2 - np.dot(t_sum, t_sum)
    return cov_ytyp / np.sqrt(cov_ytyt * cov_ypyp)


def _calculate_metrics(cnf_matrix: np.ndarray) -> dict:
    """Per-class rates from a confusion matrix (deepgrp/prediction.py:167-197)."""
    true_positive = np.diag(cnf_matrix).astype(float)
    false_positive = (cnf_matrix.sum(axis=0) - true_positive).astype(float)
    false_negative = (cnf_matrix.sum(axis=1) - true_positive).astype(float)
    true_negative = (cnf_matrix.sum() - (false_positive + false_negative + true_positive)).astype(float)
    metrics = {}
    metrics["TPR"] = true_positive / (true_positive + false_negative)
    metrics["TNR"] = true_negative / (true_negative + false_positive)
    metrics["PPV"] = true_positive / (true_positive + false_positive)
    metrics["NPV"] = true_negative / (true_negative + false_negative)
    metrics["FPR"] = false_positive / (false_positive + true_negative)
    metrics["FNR"] = false_negative / (true_positive + false_negative)
    metrics["FDR"] = false_positive / (true_positive + false_positive)
    metrics["ACC"] = (true_positive + true_negative) / \
        (true_positive + false_positive + false_negative + true_negative)
    metrics["F1"] = 2 * metrics["TPR"] * metrics["PPV"] / (metrics["TPR"] + metrics["PPV"])
    metrics["MCC"] = calculate_multiclass_matthews_cc(cnf_matrix)
    return metrics


def confusion_metrics(cnf_matrix: np.ndarray) -> dict:
    """The metrics :func:`calculate_metrics` reports for a confusion matrix (``_calculate_metrics`` + ``TotalACC``);
    a 0/0 rate is NaN, as numpy computes it, without a warning."""
    cnf_matrix = np.asarray(cnf_matrix)
    with np.errstate(divide="ignore", invalid="ignore"):
        metrics = _calculate_metrics(cnf_matrix)
        metrics["TotalACC"] = np.trace(cnf_matrix) / cnf_matrix.sum()
    return metrics


def jsonable(value):
    """``value`` with numpy arrays and scalars as JSON types; NaN becomes ``None`` (JSON ``null``)."""
    if isinstance(value, dict):
        return {k: jsonable(v) for k, v in value.items()}
    if isinstance(value, (list, tuple, np.ndarray)):
        return [jsonable(v) for v in value]
    if isinstance(value, (bool, np.bool_)):
        return bool(value)
    if isinstance(value, (int, np.integer)):
        return int(value)
    if isinstance(value, (float, np.floating)):
        return None if np.isnan(value) else float(value)
    return value


def searched_repeats(repeats, n_classes: int) -> list:
    """The repeat numbers evaluation searches for, sorted and without duplicates: ``repeats``, or ``1 .. C-1`` when it
    is None.  ``ValueError`` for a number outside ``[1, n_classes)``."""
    out = list(range(1, n_classes)) if repeats is None else sorted({int(r) for r in repeats})
    bad = [r for r in out if not 1 <= r < n_classes]
    if bad or not out:
        raise ValueError("repeat numbers must lie in [1, %d) for a %d-class model, got %s"
                         % (n_classes, n_classes, bad or "none"))
    return out


def evaluate_fasta(model: ModelWeights, raw, annotation: dict, step_size: int, batch_size: int, use_mss: bool,
                   min_mss_len: int, xdrop_len: int, repeats=None, compat: str = "reference") -> dict:
    """Score the prediction of one FASTA file (the rows ``deepgrp predict`` writes with these options) against a repeat
    annotation, on the GPU.  ``annotation``: :func:`deepgrp_b200.preprocessing.read_annotation`'s
    ``{chromosome: int64[n, 3]}``; a record's chromosome is the first word of its header.  A record's evaluated span is
    ``[startpos, startpos + length)``; a position's true class is the lowest searched repeat number among the
    annotations that cover it (``preprocess_y(...).argmax(0)``), 0 where none does; its predicted class is the label of
    the row that covers it, 0 where none does.  The file runs slice by slice (whole records, >= 8 MiB), which bounds
    device memory; no per-base array is built.  Returns ``{classes, repeats, records: [{header, chromosome, startpos,
    length, confusion, metrics}], total: {confusion, metrics}}`` with ``C x C`` int64 matrices (rows: true class).
    A blank line raises ``IndexError`` and an all-``N`` record ``ValueError``, as in ``predict``."""
    from .sharding import fasta_slices
    C = model.n_classes
    repeats = searched_repeats(repeats, C)
    wanted = np.asarray(repeats, dtype=np.int64)
    ctx = _lib.context()
    cuts, _ = fasta_slices(raw, 1)
    whole = memoryview(raw) if len(raw) else memoryview(b"")
    records = []
    none = np.zeros((0, 3), np.int64)
    for k in range(len(cuts) - 1):
        piece = whole[int(cuts[k]):int(cuts[k + 1])]
        _, recs = _predict_fasta_call(model, piece, step_size, batch_size, use_mss, min_mss_len, xdrop_len, compat)
        chroms = [header.split()[0] for header, _, _ in recs]
        lists = []
        for chrom in chroms:
            a = np.asarray(annotation.get(chrom, none), dtype=np.int64).reshape(-1, 3)
            lists.append(a[np.isin(a[:, 2], wanted)])
        ann = np.ascontiguousarray(np.concatenate(lists) if lists else none)
        ann_off = np.zeros(len(recs) + 1, np.int64)
        ann_off[1:] = np.cumsum([len(a) for a in lists])
        counts = np.zeros((max(len(recs), 1), C, C), np.int64)
        _lib.check(_lib.lib().dgrp_evaluate_last(ctx.handle, C, _lib.ptr(ann), _lib.ptr(ann_off), len(recs),
                                                 _lib.ptr(counts)))
        for (header, startpos, length), chrom, cnf in zip(recs, chroms, counts):
            records.append({"header": header, "chromosome": chrom, "startpos": startpos, "length": length,
                            "confusion": cnf, "metrics": confusion_metrics(cnf)})
    total = np.zeros((C, C), np.int64)
    for rec in records:
        total += rec["confusion"]
    return {"classes": C, "repeats": repeats, "records": records,
            "total": {"confusion": total, "metrics": confusion_metrics(total)}}


def _labels_u8(name: str, a) -> np.ndarray:
    arr = np.asarray(a)
    if arr.size and (arr.min() < 0 or arr.max() >= 16):
        raise IndexError("%s: labels must be in [0, 16) for the GPU confusion matrix" % name)
    return np.ascontiguousarray(arr.reshape(-1), dtype=np.uint8)


def confusion_matrix(truelbl: np.ndarray, predictedlbl: np.ndarray) -> np.ndarray:
    """Confusion matrix of two integer label arrays (deepgrp/prediction.py:200-218): one GPU pass
    (shared-memory counters per block).  As in the reference the matrix has
    ``max(labels) - min(labels) + 1`` rows and a label beyond that raises IndexError."""
    truelbl, predictedlbl = np.asarray(truelbl), np.asarray(predictedlbl)
    assert truelbl.size == predictedlbl.size
    n_classes = int(max(truelbl.max(), predictedlbl.max()) - min(truelbl.min(), predictedlbl.min()) + 1)
    t8, p8 = _labels_u8("truelbl", truelbl), _labels_u8("predictedlbl", predictedlbl)
    full = np.zeros(256, dtype=np.int64)
    ctx = _lib.context()
    _lib.check(_lib.lib().dgrp_confusion_matrix(ctx.handle, _lib.ptr(t8), _lib.ptr(p8), t8.size, _lib.ptr(full)))
    full = full.reshape(16, 16)
    if full[n_classes:, :].any() or full[:, n_classes:].any():
        raise IndexError("index %d is out of bounds for axis 0 with size %d"
                         % (int(max(truelbl.max(), predictedlbl.max())), n_classes))
    return full[:n_classes, :n_classes].astype(int)


def calculate_metrics(predictions_class: np.ndarray, true_class: np.ndarray):
    """(confusion matrix, metrics dict incl. TotalACC) -- deepgrp/prediction.py:221-239."""
    predictions_class, true_class = np.asarray(predictions_class), np.asarray(true_class)
    cnf_matrix = confusion_matrix(true_class, predictions_class)
    metrics = _calculate_metrics(cnf_matrix)
    metrics["TotalACC"] = np.trace(cnf_matrix) / true_class.shape[0]
    return cnf_matrix, metrics


def filter_segments(array: np.ndarray, min_len: int = 50) -> None:
    """Zero every run of one identical positive label that is shorter than `min_len`, in place
    (deepgrp/prediction.py:242-260).  Runs are found and cleared on the GPU."""
    if array.size == 0:
        return
    flat = array.reshape(-1)
    lab = _labels_u8("array", np.where(flat > 0, flat, 0))
    if not np.array_equal(lab, np.where(flat > 0, flat, 0)):
        raise ValueError("filter_segments: labels must be integers in [0, 16)")
    keep = lab.copy()
    ctx = _lib.context()
    _lib.check(_lib.lib().dgrp_filter_segments(ctx.handle, _lib.ptr(keep), keep.size, int(min_len)))
    flat[(lab > 0) & (keep == 0)] = 0

