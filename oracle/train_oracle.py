"""oracle/train_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Float64 restatement of one DeepGRP training step (deepgrp/training.py: Keras `fit` on the model of
deepgrp/model.py:293-336 with the optimiser of :202-215), used only as the checker by tests/ and, for context, by
tools/train_bench.py.  Nothing under deepgrp_b200/ imports this module.

The forward is the one of oracle.model_forward (tests/test_training_host.py checks that they agree to 1e-12 with
all-keep masks and no dropout); the gradients come from torch autograd and are pinned to central finite differences
in the same test file.
"""
from __future__ import annotations

from typing import Dict, Tuple

import numpy as np

from .oracle import COMPLEMENT

# Training (deepgrp/training.py): loss, gradients and optimiser updates, float64
# --------------------------------------------------------------------------------------------
TRAIN_PARAMS = ("kernel", "recurrent_kernel", "bias", "att_scale", "ff_kernel", "ff_bias")


def train_forward(w: Dict[str, np.ndarray], codes: np.ndarray, ymask: np.ndarray, starts: np.ndarray,
                  keep: np.ndarray, dropout: float, vecsize: int, dtype=None):
    """The training forward of a GRU model on the windows [s, s + vecsize) of a record, as torch tensors
    that autograd can differentiate: (loss, probs [B,T,C], {name: leaf tensor}).

    Input dropout: keep[b][dir][c] (0/1) scaled by 1/(1-dropout) multiplies channel c of the input the GRU sees
    (dir 0: x, dir 1: the reverse complement).  Loss: Keras categorical_crossentropy on probabilities -- p / sum p,
    clipped to [1e-7, 1-1e-7], -sum_c y_c log p_c -- averaged over every position; y_c = bit c of ymask.

    ``dtype`` (default torch.float64) is the torch type of every tensor.  With torch.float32 the same math runs in
    float32 on the CPU: its distance from the float64 result measures the float32 rounding noise of a shape, the
    yardstick for the tolerance of a comparison with the fp32 GPU kernels."""
    import torch
    dt = torch.float64 if dtype is None else dtype
    prm = {k: torch.tensor(np.asarray(w[k], dtype=np.float64), dtype=dt, requires_grad=True)
           for k in TRAIN_PARAMS if w.get(k) is not None}
    T = int(vecsize)
    starts = np.asarray(starts, dtype=np.int64)
    idx = starts[:, None] + np.arange(T)[None, :]
    x = torch.nn.functional.one_hot(torch.from_numpy(np.asarray(codes, np.int64)[idx]), 5).to(dt)
    x_rc = x.flip(1)[:, :, COMPLEMENT]
    keep = (torch.from_numpy(np.asarray(keep, dtype=np.float64)) / (1.0 - dropout)).to(dt)
    units = prm["recurrent_kernel"].shape[0]

    def gru(inp):
        h = torch.zeros(inp.shape[0], units, dtype=dt)
        seq = []
        for t in range(T):
            mx = inp[:, t, :] @ prm["kernel"] + prm["bias"][0]
            mh = h @ prm["recurrent_kernel"] + prm["bias"][1]
            z = torch.sigmoid(mx[:, :units] + mh[:, :units])
            r = torch.sigmoid(mx[:, units:2 * units] + mh[:, units:2 * units])
            hh = torch.tanh(mx[:, 2 * units:] + r * mh[:, 2 * units:])
            h = z * h + (1 - z) * hh
            seq.append(h)
        return torch.stack(seq, 1), h

    fwd, hf = gru(x * keep[:, None, 0, :])
    rev, hr = gru(x_rc * keep[:, None, 1, :])
    avg = (fwd + rev) * 0.5
    if "att_scale" in prm:
        q = (hf + hr) * 0.5
        scores = (prm["att_scale"] * torch.tanh(q[:, None, :] + avg)).sum(-1)
        att = torch.softmax(scores, dim=1)
        ctx = torch.einsum("bt,btu->bu", att, avg)
        feat = torch.cat([ctx[:, None, :].expand(-1, T, -1), avg], dim=2)
    else:
        feat = avg
    probs = torch.softmax(feat @ prm["ff_kernel"] + prm["ff_bias"], dim=2)
    n_classes = probs.shape[2]
    ybits = np.asarray(ymask, np.int64)[idx][:, :, None] >> np.arange(n_classes)[None, None, :]
    y = torch.from_numpy((ybits & 1).astype(np.float64)).to(dt)
    p = probs / probs.sum(-1, keepdim=True)
    p = torch.clamp(p, 1e-7, 1 - 1e-7)
    loss = -(y * torch.log(p)).sum(-1).mean()
    return loss, probs, prm


def train_loss_and_grads(w: Dict[str, np.ndarray], codes: np.ndarray, ymask: np.ndarray, starts: np.ndarray,
                         keep: np.ndarray, dropout: float, vecsize: int, dtype=None):
    """(loss, {name: gradient}, probs [B,T,C]) of one training batch (see `train_forward`), as numpy arrays of
    ``dtype`` (default float64)."""
    loss, probs, prm = train_forward(w, codes, ymask, starts, keep, dropout, vecsize, dtype)
    loss.backward()
    return float(loss.item()), {k: v.grad.numpy().copy() for k, v in prm.items()}, probs.detach().numpy()


def optimizer_step(name: str, w: np.ndarray, g: np.ndarray, state: Dict[str, np.ndarray], step: int,
                   learning_rate: float = 1e-3, rho: float = 0.9, momentum: float = 0.9,
                   epsilon: float = 1e-10) -> Tuple[np.ndarray, Dict[str, np.ndarray]]:
    """One update of one weight array, float64: "RMSprop" (momentum > 0: TF ApplyRMSProp; momentum 0: Keras'
    w - lr g / (sqrt(ms) + eps)) or "Adam" (Keras, beta1 0.9, beta2 0.999; `step` counts from 1).  `state` holds
    ms / mom or m / v (missing entries start at zero).  Returns (new w, new state)."""
    w = np.asarray(w, np.float64)
    g = np.asarray(g, np.float64)
    zero = np.zeros_like(w)
    if name == "RMSprop":
        ms = rho * state.get("ms", zero) + (1 - rho) * g * g
        if momentum > 0:
            mom = momentum * state.get("mom", zero) + learning_rate * g / np.sqrt(ms + epsilon)
            return w - mom, {"ms": ms, "mom": mom}
        return w - learning_rate * g / (np.sqrt(ms) + epsilon), {"ms": ms}
    if name == "Adam":
        b1, b2 = 0.9, 0.999
        m = b1 * state.get("m", zero) + (1 - b1) * g
        v = b2 * state.get("v", zero) + (1 - b2) * g * g
        lr_t = learning_rate * np.sqrt(1 - b2 ** step) / (1 - b1 ** step)
        return w - lr_t * m / (np.sqrt(v) + epsilon), {"m": m, "v": v}
    raise ValueError("unknown optimizer %r" % name)
