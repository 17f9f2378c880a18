"""deepgrp_b200.model -- hyper-parameters and weight container for the prediction path.

Mirrors the parts of the reference's ``deepgrp/model.py`` that the prediction path touches:

* ``Options`` (reference ``deepgrp/model.py:28-199``): the same attribute names and defaults, the
  ``gru_units``/``gru_dropout`` legacy aliases, dict and TOML round trips.
* ``create_model(options)`` (reference ``deepgrp/model.py:293-336``): instead of a compiled Keras
  graph it returns a ``ModelWeights`` with Keras' default initialisers (GlorotUniform kernels,
  Orthogonal recurrent kernel, zero biases), i.e. a random-init model of the same architecture.
  The forward topology itself lives in the CUDA kernels (``csrc/forward.cu``).
* ``ModelWeights`` stands where ``keras.Model`` stood: it has ``input_shape``/``output_shape``
  (used by the CLI, reference ``deepgrp/__main__.py:270`` and ``:75``) and ``predict_on_batch``.

The optimiser that ``_get_optimizer`` builds in the reference is chosen by ``deepgrp_b200.training`` from
``Options.optimizer`` (``"RMSprop"`` or ``"Adam"``) and runs on the GPU; ``create_logdir`` has no counterpart (training
writes into the ``logdir`` it is given).
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, TextIO, Tuple, Union

import numpy as np

COMPLEMENT_INDICES = [3, 2, 1, 0, 4]     # reference deepgrp/model.py:233-237 (_get_dna_encoding)

_DEFAULTS: Dict[str, Any] = dict(
    # general (reference deepgrp/model.py:84-99)
    project_root_dir=".", repeats_to_search=[1, 2, 3, 4], vecsize=150, n_epochs=200,
    n_batches=250, early_stopping_th=10, batch_size=256, repeat_probability=0.3,
    # optimiser (:103-112) -- used by deepgrp_b200.training
    optimizer="RMSprop", learning_rate=0.001, momentum=0.9, rho=0.9, epsilon=1e-10,
    # network (:116-123)
    rnn="GRU", units=32, dropout=0.25, attention=False,
    # MSS (:127-129)
    min_mss_len=50, xdrop_len=50,
)


class Options:
    """Attribute bag of hyper-parameters (reference ``deepgrp/model.py:28-199``)."""

    def __init__(self, **kwargs) -> None:
        for key, value in _DEFAULTS.items():
            setattr(self, key, list(value) if isinstance(value, list) else value)
        self.__dict__.update(kwargs)
        self._fold_legacy_names()

    def _fold_legacy_names(self) -> None:
        # `gru_units` / `gru_dropout` are accepted and folded into units / dropout (:131-144)
        for old, new in (("gru_units", "units"), ("gru_dropout", "dropout")):
            value = self.__dict__.pop(old, None)
            if value:
                self.__dict__[new] = value

    def __setitem__(self, key: str, item: Union[float, int, str]) -> None:
        self.__dict__[key.replace("gru_", "")] = item

    def __getitem__(self, key: str) -> Union[float, int, str]:
        return self.__dict__[key.replace("gru_", "")]

    def __str__(self) -> str:
        return str(self.__dict__)

    def todict(self) -> Dict[str, Any]:
        return self.__dict__.copy()

    def fromdict(self, dictionary: Dict[str, Any]) -> None:
        self.__dict__.update(dictionary)
        self._fold_legacy_names()

    @classmethod
    def from_toml(cls, file: TextIO) -> "Options":
        if not hasattr(file, "read"):
            raise TypeError("from_toml expects an open file")
        text = file.read()
        try:
            import tomllib
            return cls(**tomllib.loads(text))
        except ModuleNotFoundError:          # pragma: no cover  (python < 3.11)
            import toml
            return cls(**toml.loads(text))

    def to_toml(self, file: TextIO) -> None:
        if not hasattr(file, "write"):
            raise TypeError("to_toml expects a writable file")

        def fmt(v):
            if isinstance(v, bool):
                return "true" if v else "false"
            if isinstance(v, str):
                return '"' + v.replace("\\", "\\\\").replace('"', '\\"') + '"'
            if isinstance(v, (list, tuple)):
                return "[ " + ", ".join(fmt(x) for x in v) + ",]"
            return repr(v)

        for key, value in self.__dict__.items():
            file.write("{} = {}\n".format(key, fmt(value)))


class ModelWeights:
    """Host-side weights of one DeepGRP model (what the Keras HDF5 file holds).

    Arrays (float32, C-contiguous), named after the Keras variables they come from:
      kernel            [5, G*U]  BGRU/gru_cell/kernel           (G = 3 gates z,r,h for GRU;
      recurrent_kernel  [U, G*U]  BGRU/gru_cell/recurrent_kernel      4 gates i,f,c,o for LSTM)
      bias              [2, G*U]  BGRU/gru_cell/bias  (row 0 input, row 1 recurrent; LSTM: [1,4U])
      att_scale         [U]       additive_attention/scale       (None without attention)
      ff_kernel         [F, C]    FF/kernel   (F = 2U with attention, else U)
      ff_bias           [C]       FF/bias
    """

    def __init__(self, vecsize: int, units: int, kernel, recurrent_kernel, bias, ff_kernel,
                 ff_bias, att_scale=None, rnn: str = "GRU") -> None:
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        self.vecsize = int(vecsize)
        self.units = int(units)
        self.rnn = rnn
        self.kernel = f32(kernel)
        self.recurrent_kernel = f32(recurrent_kernel)
        self.bias = f32(bias)
        self.att_scale = None if att_scale is None else f32(att_scale)
        self.ff_kernel = f32(ff_kernel)
        self.ff_bias = f32(ff_bias)
        gates = 4 if rnn == "LSTM" else 3
        u = self.units
        if self.kernel.shape != (5, gates * u):
            raise ValueError("kernel must be [5, %d], got %s" % (gates * u, self.kernel.shape))
        if self.recurrent_kernel.shape != (u, gates * u):
            raise ValueError("recurrent_kernel must be [%d, %d]" % (u, gates * u))
        if self.bias.ndim == 1:
            self.bias = self.bias.reshape(1, -1)
        feat = 2 * u if self.attention else u
        if self.ff_kernel.shape[0] != feat:
            raise ValueError("FF kernel rows %d != %d" % (self.ff_kernel.shape[0], feat))
        self._device_handles: Dict[int, Any] = {}

    @property
    def attention(self) -> bool:
        return self.att_scale is not None

    @property
    def n_classes(self) -> int:
        return int(self.ff_kernel.shape[1])

    # keras.Model look-alikes used by the reference CLI
    @property
    def input_shape(self) -> Tuple[Optional[int], int, int]:
        return (None, self.vecsize, 5)

    @property
    def output_shape(self) -> Tuple[Optional[int], int, int]:
        return (None, self.vecsize, self.n_classes)

    def as_dict(self) -> Dict[str, np.ndarray]:
        d = dict(kernel=self.kernel, recurrent_kernel=self.recurrent_kernel, bias=self.bias,
                 ff_kernel=self.ff_kernel, ff_bias=self.ff_bias)
        if self.att_scale is not None:
            d["att_scale"] = self.att_scale
        return d

    def scaled(self, factor: float) -> "ModelWeights":
        """Same shapes with every weight multiplied by `factor` (SURVEY.md §8d second weight set)."""
        return ModelWeights(self.vecsize, self.units, self.kernel * factor,
                            self.recurrent_kernel * factor, self.bias * factor,
                            self.ff_kernel * factor, self.ff_bias * factor,
                            None if self.att_scale is None else self.att_scale * factor, self.rnn)

    def device_handle(self, ctx):
        """``dgrp_model*`` of these weights on the context's GPU (uploaded on first use)."""
        import ctypes
        from . import _lib
        key = ctx.device
        handle = self._device_handles.get(key)
        if handle is None:
            if self.rnn not in ("GRU", "LSTM"):
                raise NotImplementedError("rnn must be 'GRU' or 'LSTM'")
            handle = ctypes.c_void_p()
            _lib.check(_lib.lib().dgrp_model_create(
                ctx.handle, 1 if self.rnn == "LSTM" else 0, self.vecsize, self.units, self.n_classes, _lib.ptr(self.kernel),
                _lib.ptr(self.recurrent_kernel), _lib.ptr(self.bias), _lib.ptr(self.att_scale),
                _lib.ptr(self.ff_kernel), _lib.ptr(self.ff_bias), ctypes.byref(handle)))
            self._device_handles[key] = handle
            self._handle_vecsize = self.vecsize
        elif getattr(self, "_handle_vecsize", self.vecsize) != self.vecsize:
            self.release()
            return self.device_handle(ctx)
        return handle

    def release(self) -> None:
        from . import _lib
        for handle in self._device_handles.values():
            _lib.lib().dgrp_model_destroy(handle)
        self._device_handles = {}

    def predict_on_batch(self, batch):
        """keras.Model.predict_on_batch stand-in: float32[B,T,5] one-hot windows -> float32[B,T,C]
        through the CUDA forward (no CPU fallback)."""
        from . import prediction
        return prediction.forward_windows(self, batch)

    def save_npz(self, path: str) -> None:
        np.savez(path, vecsize=self.vecsize, units=self.units, rnn=self.rnn, **self.as_dict())

    @classmethod
    def load_npz(cls, path: str) -> "ModelWeights":
        z = np.load(path, allow_pickle=False)
        return cls(int(z["vecsize"]), int(z["units"]), z["kernel"], z["recurrent_kernel"],
                   z["bias"], z["ff_kernel"], z["ff_bias"],
                   z["att_scale"] if "att_scale" in z.files else None,
                   str(z["rnn"]) if "rnn" in z.files else "GRU")


def load_model(path: str) -> ModelWeights:
    """Stands where ``tf.keras.models.load_model`` stood (reference ``deepgrp/__main__.py:264-269``):
    reads a Keras HDF5 model file (``.hdf5``/``.h5``) or the ``.npz`` side format."""
    if str(path).endswith(".npz"):
        return ModelWeights.load_npz(path)
    from . import hdf5
    return hdf5.load_keras_model(path)


def _glorot_uniform(rng: np.random.Generator, shape, fan_in: int, fan_out: int) -> np.ndarray:
    limit = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-limit, limit, size=shape).astype(np.float32)


def _orthogonal(rng: np.random.Generator, rows: int, cols: int) -> np.ndarray:
    """Keras Orthogonal initialiser: QR of a normal [max,min] matrix, sign-fixed by diag(R)."""
    flat = (max(rows, cols), min(rows, cols))
    q, r = np.linalg.qr(rng.normal(size=flat))
    q = q * np.sign(np.diag(r))
    if rows < cols:
        q = q.T
    return np.ascontiguousarray(q[:rows, :cols], dtype=np.float32)


def random_weights(vecsize: int, units: int, attention: bool = True, n_classes: int = 5,
                   seed: int = 0, rnn: str = "GRU") -> ModelWeights:
    """Random-init weights of the architecture `create_model` builds (Keras default initialisers;
    SURVEY.md §8d fixes seed 0 for the benchmark models)."""
    rng = np.random.default_rng(seed)
    gates = 4 if rnn == "LSTM" else 3
    kernel = _glorot_uniform(rng, (5, gates * units), 5, gates * units)
    recurrent = _orthogonal(rng, units, gates * units)
    if rnn == "LSTM":
        bias = np.zeros((1, gates * units), np.float32)
        bias[0, units:2 * units] = 1.0                      # unit_forget_bias=True
    else:
        bias = np.zeros((2, gates * units), np.float32)
    use_att = attention and rnn != "LSTM"                   # reference deepgrp/model.py:308
    scale = _glorot_uniform(rng, (units,), units, units) if use_att else None
    feat = 2 * units if use_att else units
    ff_kernel = _glorot_uniform(rng, (feat, n_classes), feat, n_classes)
    ff_bias = np.zeros(n_classes, np.float32)
    return ModelWeights(vecsize, units, kernel, recurrent, bias, ff_kernel, ff_bias, scale, rnn)


def create_model(options: Options, seed: int = 0) -> ModelWeights:
    """Reference ``deepgrp/model.py:293-336``: a fresh (random-init) model for `options`."""
    return random_weights(options.vecsize, options.units, bool(options.attention),
                          len(options.repeats_to_search) + 1, seed=seed, rnn=options.rnn)
