"""deepgrp_b200.training -- training of DeepGRP models on the GPU (reference ``deepgrp/training.py``).

The reference builds two ``tf.data`` datasets from ``fetch_batch`` and calls ``keras.Model.fit``.  Here the same
loop runs through the CUDA trainer of ``csrc/train.cu`` (``dgrp_train_*``): the windows of a batch are never
materialised -- the sampler hands the GPU window starts and input-dropout masks, the record's base codes and label
masks are uploaded once -- and the forward, backward and optimiser update are CUDA kernels (fp32, bit-reproducible
on one GPU).  Supported: ``rnn="GRU"`` with ``units <= 64`` and 2 to 5 classes, the models prediction runs; anything
else is refused when the ``Trainer`` is created, before the first step.

Rules of this port where the reference's exact behaviour is not available (README.md lists them):

* Sampler (``BatchSampler``): per window, with probability ``repeat_probability`` a class is drawn uniformly among
  the ``repeats_to_search`` that occur in the record, then a uniform position of that class, and the window starts
  ``U[0, vecsize)`` bases before it, clipped to the record; otherwise the start is uniform.  Input-dropout keeps are
  Bernoulli(1 - dropout) per window, direction and channel, from the same seeded generator.
* Validation: ``n_batches`` batches of ``batch_size`` windows drawn once (same rule, generator seeded from ``seed``),
  evaluated without dropout after every epoch.
* Early stopping after ``early_stopping_th`` epochs without a lower validation loss; the best weights are written to
  ``logdir/best.hdf5`` whenever they improve and are the model's weights when ``training`` returns.
"""
from __future__ import annotations

import ctypes
import os
import time
from typing import Dict, Iterator, List, NamedTuple, Optional, Tuple

import numpy as np

from . import _lib
from .model import ModelWeights, Options

OPTIMIZERS = {"RMSprop": _lib.OPT_RMSPROP, "Adam": _lib.OPT_ADAM}
_ARRAYS = ("kernel", "recurrent_kernel", "bias", "att_scale", "ff_kernel", "ff_bias")


def onehot_to_codes(fwd: np.ndarray) -> np.ndarray:
    """int8[5, L] one-hot matrix (rows A, C, G, T, N, as ``preprocess_sequence`` writes it) -> uint8[L] base codes.
    A column that is not exactly one-hot is a ``ValueError``."""
    fwd = np.asarray(fwd)
    if fwd.ndim != 2 or fwd.shape[0] != 5:
        raise ValueError("expected a one-hot matrix of shape [5, L], got %s" % (fwd.shape,))
    bad = ~(((fwd == 0) | (fwd == 1)).all(axis=0) & (fwd.sum(axis=0) == 1))
    if bad.any():
        raise ValueError("column %d of the one-hot matrix is not one-hot: %s"
                         % (int(np.argmax(bad)), fwd[:, int(np.argmax(bad))].tolist()))
    return np.ascontiguousarray(np.argmax(fwd, axis=0), dtype=np.uint8)


def labels_to_mask(truelbl: np.ndarray) -> np.ndarray:
    """int8[C, L] label matrix of ``preprocess_y`` (several rows set where annotations overlap) -> uint8[L] with bit
    c set where row c is set."""
    y = np.asarray(truelbl)
    if y.ndim != 2 or not 1 <= y.shape[0] <= 8:
        raise ValueError("expected a label matrix of shape [C <= 8, L], got %s" % (y.shape,))
    mask = np.zeros(y.shape[1], dtype=np.uint8)
    for c in range(y.shape[0]):
        mask |= (y[c] != 0).astype(np.uint8) << c
    return mask


class Draw(NamedTuple):
    starts: np.ndarray        # int64[B]   window starts
    keep: np.ndarray          # uint8[B, 2, 5]  input-dropout keeps (direction 0: x, 1: reverse complement)
    repeat_class: np.ndarray  # int64[B]   class row a window was drawn around, -1 for a uniform window


class BatchSampler:
    """The window sampler of ``fetch_batch`` on one record's label matrix ``y_data`` (int8[C, L])."""

    def __init__(self, y_data: np.ndarray, options: Options):
        y = np.asarray(y_data)
        self.length = int(y.shape[1])
        self.vecsize = int(options.vecsize)
        if self.length < self.vecsize:
            raise ValueError("record length %d is shorter than vecsize %d" % (self.length, self.vecsize))
        self.batch_size = int(options.batch_size)
        self.repeat_probability = float(options.repeat_probability)
        self.dropout = float(options.dropout)
        self.classes = [int(r) for r in options.repeats_to_search if 0 <= int(r) < y.shape[0] and y[int(r)].any()]
        self.positions = [np.flatnonzero(y[r]) for r in self.classes]

    def draw(self, rng: np.random.Generator, batch_size: Optional[int] = None) -> Draw:
        n = self.batch_size if batch_size is None else int(batch_size)
        T, last = self.vecsize, self.length - self.vecsize
        repeat = rng.random(n) < self.repeat_probability
        which = rng.integers(0, max(len(self.classes), 1), size=n)
        frac = rng.random(n)
        offset = rng.integers(0, T, size=n)
        starts = rng.integers(0, last + 1, size=n).astype(np.int64)
        repeat_class = np.full(n, -1, dtype=np.int64)
        if self.classes:
            for i, (cls, pos) in enumerate(zip(self.classes, self.positions)):
                sel = repeat & (which == i)
                centre = pos[(frac[sel] * pos.size).astype(np.int64)]
                starts[sel] = np.clip(centre - offset[sel], 0, last)
                repeat_class[sel] = cls
        keep = (rng.random((n, 2, 5)) < 1.0 - self.dropout).astype(np.uint8)
        return Draw(starts, keep, repeat_class)


def fetch_batch(x_data: np.ndarray, y_data: np.ndarray, options: Options,
                rng: np.random.Generator) -> Iterator[Tuple[np.ndarray, np.ndarray]]:
    """Reference ``deepgrp/training.py:84-132``: endless batches of float32 windows [B, T, 5] of the one-hot matrix
    ``x_data`` (int8[5, L]) and their targets [B, T, C] from ``y_data`` (int8[C, L]), drawn by ``BatchSampler``.
    (``training`` draws the same starts and masks without building these arrays.)"""
    sampler = BatchSampler(y_data, options)
    x_t, y_t = np.asarray(x_data).T, np.asarray(y_data).T
    T = sampler.vecsize
    while True:
        d = sampler.draw(rng)
        yield (np.stack([x_t[s:s + T] for s in d.starts]).astype(np.float32),
               np.stack([y_t[s:s + T] for s in d.starts]).astype(np.float32))


class Trainer:
    """A model, its optimiser state and its records on the GPU (``dgrp_trainer``)."""

    def __init__(self, model: ModelWeights, options: Options, ctx: Optional[_lib.Context] = None):
        if options.optimizer not in OPTIMIZERS:
            raise ValueError("optimizer must be one of %s, got %r" % (sorted(OPTIMIZERS), options.optimizer))
        self.ctx = ctx or _lib.context()
        self.vecsize, self.units, self.n_classes = model.vecsize, model.units, model.n_classes
        self.attention = model.attention
        self.rnn = model.rnn
        self.optimizer = options.optimizer
        handle = ctypes.c_void_p()
        _lib.check(_lib.lib().dgrp_train_create(
            self.ctx.handle, 1 if model.rnn == "LSTM" else 0, model.vecsize, model.units, model.n_classes,
            1 if model.attention else 0, _lib.ptr(model.kernel), _lib.ptr(model.recurrent_kernel),
            _lib.ptr(model.bias), _lib.ptr(model.att_scale), _lib.ptr(model.ff_kernel), _lib.ptr(model.ff_bias),
            OPTIMIZERS[options.optimizer], float(options.learning_rate), float(options.rho),
            float(options.momentum), float(options.epsilon), float(options.dropout), ctypes.byref(handle)))
        self.handle = handle

    def set_data(self, which: int, codes: np.ndarray, ymask: np.ndarray) -> None:
        """Upload a record: which 0 = training, 1 = validation; uint8 base codes and label masks of equal length."""
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        ymask = np.ascontiguousarray(ymask, dtype=np.uint8)
        if codes.shape != ymask.shape or codes.ndim != 1:
            raise ValueError("codes and ymask must be 1-D arrays of one length")
        _lib.check(_lib.lib().dgrp_train_set_data(self.handle, int(which), _lib.ptr(codes), _lib.ptr(ymask),
                                                  codes.size))

    def step(self, starts: np.ndarray, keep: np.ndarray) -> float:
        """One optimiser step on the training windows at ``starts`` with input-dropout keeps uint8[n, 2, 5];
        returns the batch's loss before the update."""
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        keep = np.ascontiguousarray(keep, dtype=np.uint8)
        if keep.shape != (starts.size, 2, 5):
            raise ValueError("keep must have shape [%d, 2, 5], got %s" % (starts.size, keep.shape))
        loss = ctypes.c_float()
        _lib.check(_lib.lib().dgrp_train_step(self.handle, _lib.ptr(starts), _lib.ptr(keep), starts.size,
                                              ctypes.byref(loss)))
        return float(loss.value)

    def evaluate(self, which: int, starts: np.ndarray, probs: bool = False):
        """Mean loss of the windows at ``starts`` of record ``which`` without dropout and update; with ``probs``
        also their probabilities float32[n, T, C]."""
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        out = np.zeros((starts.size, self.vecsize, self.n_classes), np.float32) if probs else None
        loss = ctypes.c_float()
        _lib.check(_lib.lib().dgrp_train_eval(self.handle, int(which), _lib.ptr(starts), starts.size,
                                              ctypes.byref(loss), _lib.ptr(out)))
        return (float(loss.value), out) if probs else float(loss.value)

    def _fetch(self, fn) -> Dict[str, np.ndarray]:
        u, c = self.units, self.n_classes
        f = 2 * u if self.attention else u
        out = dict(kernel=np.zeros((5, 3 * u), np.float32), recurrent_kernel=np.zeros((u, 3 * u), np.float32),
                   bias=np.zeros((2, 3 * u), np.float32),
                   att_scale=np.zeros(u, np.float32) if self.attention else None,
                   ff_kernel=np.zeros((f, c), np.float32), ff_bias=np.zeros(c, np.float32))
        _lib.check(fn(self.handle, *[_lib.ptr(out[k]) for k in _ARRAYS]))
        return out

    def weights(self) -> Dict[str, np.ndarray]:
        """Current weights in the Keras layouts (``att_scale`` None without attention)."""
        return self._fetch(_lib.lib().dgrp_train_get_weights)

    def grads(self) -> Dict[str, np.ndarray]:
        """Gradients of the last step, before its update, in the layouts of ``weights``."""
        return self._fetch(_lib.lib().dgrp_train_get_grads)

    def model(self) -> ModelWeights:
        w = self.weights()
        return ModelWeights(self.vecsize, self.units, w["kernel"], w["recurrent_kernel"], w["bias"],
                            w["ff_kernel"], w["ff_bias"], w["att_scale"], self.rnn)

    def timings(self) -> Dict[str, float]:
        """Device milliseconds of the last step's phases."""
        out = np.zeros(5, np.float32)
        _lib.check(_lib.lib().dgrp_train_timings(self.handle, _lib.ptr(out)))
        return dict(zip(("forward", "head", "bptt", "reduction", "update"), map(float, out)))

    def close(self) -> None:
        if getattr(self, "handle", None):
            _lib.lib().dgrp_train_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # interpreter shutdown
            pass


def training(data, options: Options, model: ModelWeights, logdir, seed: int = 0) -> List[Tuple[int, float, float, float]]:
    """Reference ``deepgrp/training.py:15-73``: trains ``model`` in place on ``data = (train, validation)``
    (``preprocessing.Data`` tuples: one-hot int8[5, L] and labels int8[C, L]) for up to ``n_epochs`` epochs of
    ``n_batches`` steps.  Writes ``logdir/best.hdf5`` at every new best validation loss and one line per epoch to
    ``logdir/history.tsv``; returns the history rows (epoch, train loss, validation loss, seconds)."""
    from . import hdf5
    train, valid = data
    os.makedirs(logdir, exist_ok=True)
    rng = np.random.default_rng(seed)
    sampler = BatchSampler(train.truelbl, options)
    val_sampler = BatchSampler(valid.truelbl, options)
    val_rng = np.random.default_rng([seed, 1])
    val_starts = np.concatenate([val_sampler.draw(val_rng).starts for _ in range(int(options.n_batches))])
    trainer = Trainer(model, options)
    history: List[Tuple[int, float, float, float]] = []
    best_weights = None
    try:
        trainer.set_data(0, onehot_to_codes(train.fwd), labels_to_mask(train.truelbl))
        trainer.set_data(1, onehot_to_codes(valid.fwd), labels_to_mask(valid.truelbl))
        best, waited = np.inf, 0
        hist_path = os.path.join(logdir, "history.tsv")
        with open(hist_path, "w") as fh:
            fh.write("epoch\ttrain_loss\tval_loss\tseconds\n")
        for epoch in range(1, int(options.n_epochs) + 1):
            t0 = time.perf_counter()
            losses = [trainer.step(d.starts, d.keep)
                      for d in (sampler.draw(rng) for _ in range(int(options.n_batches)))]
            val_loss = trainer.evaluate(1, val_starts)
            seconds = time.perf_counter() - t0
            row = (epoch, float(np.mean(losses)), val_loss, seconds)
            history.append(row)
            with open(hist_path, "a") as fh:
                fh.write("%d\t%.6g\t%.6g\t%.3f\n" % row)
            if val_loss < best:
                best, waited = val_loss, 0
                best_weights = trainer.model()
                hdf5.save_keras_model(os.path.join(logdir, "best.hdf5"), best_weights)
            else:
                waited += 1
                if waited >= int(options.early_stopping_th):
                    break
    finally:
        trainer.close()
    if best_weights is not None:
        for name in _ARRAYS:
            setattr(model, name, getattr(best_weights, name))
    model.release()     # device handles of the old weights must not be reused
    return history
