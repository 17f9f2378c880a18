"""Training on the GPU (csrc/train.cu through dgrp_train_*): gradients and updates against the float64 oracle,
the trainer's forward against inference, determinism, a model that learns planted repeats, the CLI end to end and
the refusals.

Tolerances: a comparison with the float64 oracle keeps a fixed bound (1e-5 for losses, 1e-4 relative for
gradients) unless the float32 rounding noise of its shape is larger.  That noise is measured, not guessed: the same
math run in float32 on the CPU (`train_oracle`, dtype=torch.float32) is `e32` away from float64, and the bound
becomes max(fixed, 8 e32)."""
import os

import numpy as np
import pytest

from deepgrp_b200 import _lib
from deepgrp_b200 import __main__ as cli
from deepgrp_b200 import model as dgmodel
from deepgrp_b200 import prediction as dgpred
from deepgrp_b200 import preprocessing as dgprep
from deepgrp_b200 import training as dgtrain
from oracle import train_oracle

pytestmark = pytest.mark.gpu
NAMES = ("kernel", "recurrent_kernel", "bias", "att_scale", "ff_kernel", "ff_bias")


def _record(length, seed, n_classes=5):
    """Random base codes (a few N) and a multi-hot label mask with overlapping annotations."""
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, 4, size=length).astype(np.uint8)
    codes[rng.random(length) < 0.02] = 4
    y = np.zeros((n_classes, length), np.int8)
    for c in range(1, n_classes):
        for _ in range(max(3, length // 200)):
            a = int(rng.integers(0, length - 10))
            y[c, a:a + int(rng.integers(5, 80))] = 1
    y[0, ~y[1:].any(axis=0)] = 1
    return codes, dgtrain.labels_to_mask(y), y


def _model(T, U, attention, seed, C=5):
    w = dgmodel.random_weights(T, U, attention=attention, n_classes=C, seed=seed).scaled(2.0)
    rng = np.random.default_rng(seed + 100)
    w.bias = (rng.normal(size=w.bias.shape) * 0.1).astype(np.float32)
    w.ff_bias = (rng.normal(size=w.ff_bias.shape) * 0.1).astype(np.float32)
    return w


def _trainer(gpu_ctx, w, codes, ymask, **options):
    tr = dgtrain.Trainer(w, dgmodel.Options(**options), gpu_ctx)
    tr.set_data(0, codes, ymask)
    tr.set_data(1, codes, ymask)
    return tr


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / max(np.linalg.norm(b), 1e-30))


def _w64(w):
    d = w if isinstance(w, dict) else w.as_dict()
    return {k: (None if d.get(k) is None else np.asarray(d[k], np.float64)) for k in NAMES}


def _parts(grads, ref):
    """(label, got, ref) of every gradient; bias rows separately: row 0 (input) and row 1 (recurrent) come from
    different sums."""
    for name, g in ref.items():
        if name == "bias":
            yield "bias0", grads[name][0], g[0]
            yield "bias1", grads[name][1], g[1]
        else:
            yield name, grads[name], g


def _e32(w64, codes, ymask, starts, keep, dropout, T, loss_o, grads_o, probs_o):
    """The float32 rounding noise of a batch: the float32 oracle's distance from the float64 one -- relative for the
    loss and each gradient, absolute (max) for the probabilities."""
    import torch
    l32, g32, p32 = train_oracle.train_loss_and_grads(w64, codes, ymask, starts, keep, dropout, T,
                                                      dtype=torch.float32)
    e = {"loss": abs(l32 - loss_o) / abs(loss_o), "probs": float(np.abs(p32 - probs_o).max())}
    e.update({label: _rel(got, ref) for label, got, ref in _parts(g32, grads_o)})
    worst = max((k for k in e if k != "probs"), key=e.get)
    print("e32 (n=%d, T=%d, U=%d, C=%d): largest %.3g (%s)" % (len(starts), T, w64["recurrent_kernel"].shape[0],
                                                             w64["ff_bias"].size, e[worst], worst))
    return e


def _check_step(loss, grads, w64, codes, ymask, starts, keep, dropout, T):
    """A step's loss and gradients against the float64 oracle, within max(fixed bound, 8 e32)."""
    loss_o, grads_o, probs_o = train_oracle.train_loss_and_grads(w64, codes, ymask, starts, keep, dropout, T)
    e = _e32(w64, codes, ymask, starts, keep, dropout, T, loss_o, grads_o, probs_o)
    assert abs(loss - loss_o) <= max(1e-5, 8 * e["loss"]) * abs(loss_o), (loss, loss_o)
    assert set(grads_o) == {k for k in NAMES if grads[k] is not None}
    for label, got, ref in _parts(grads, grads_o):
        assert _rel(got, ref) <= max(1e-4, 8 * e[label]), (label, _rel(got, ref), e[label])


def _max_vecsize(gpu_ctx, U, C, attention):
    """The largest vecsize a trainer accepts for this model shape, by bisection on creation (a host-side check of
    the head kernel's shared memory; no kernel runs)."""
    def accepted(T):
        try:
            dgtrain.Trainer(dgmodel.random_weights(T, U, attention=attention, n_classes=C), dgmodel.Options(),
                            gpu_ctx).close()
            return True
        except _lib.DeepgrpError as e:
            assert e.code == _lib.E_UNSUPPORTED and "shared memory" in str(e), e
            return False
    lo, hi = 1, 1 << 16
    assert accepted(lo) and not accepted(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if accepted(mid) else (lo, mid)
    return lo


# masks: "random" keeps at dropout 0.25; "keep" all ones at dropout 0.25; "nodrop" all ones at dropout 0 (keep scale
# exactly 1); "holes" dropout 0.5, windows 1 and 2 lose a whole direction and window 3 is all N.
# T: "max" is the largest vecsize the trainer accepts for the shape; "sm" / "sm+1" make the reduction's item count
# 2nT (n = 1) equal to its 2 * sm_count chunks, or one row more so that the trailing chunks are empty.
@pytest.mark.parametrize("T,U,attention,n,masks,C", [
    (150, 32, True, 3, "random", 5),
    (342, 60, True, 256, "random", 5),
    (40, 16, False, 1, "keep", 5),
    (40, 16, False, 3, "random", 5),
    (7, 1, True, 3, "random", 5),
    (64, 64, True, 3, "keep", 5),
    (150, 32, True, 256, "keep", 5),
    (1, 16, True, 5, "random", 5),            # attention over a single score; 10 rows: the last CTA holds 2
    (40, 33, True, 3, "random", 2),           # a tail in the head's 32-lane unit loops; two classes
    (257, 33, True, 3, "random", 5),          # crosses the head's 256-thread time loops
    ("max", 64, True, 1, "keep", 5),
    ("sm", 16, True, 1, "random", 5),
    ("sm+1", 16, True, 1, "random", 5),
    (40, 16, True, 4, "nodrop", 5),
    (40, 16, True, 6, "holes", 3),
])
def test_gradients_match_the_float64_oracle(gpu_ctx, T, U, attention, n, masks, C):
    if T == "max":
        T = _max_vecsize(gpu_ctx, U, C, attention)
    elif T in ("sm", "sm+1"):
        T = gpu_ctx.get_int("sm_count") + (T == "sm+1")
    L = max(4 * T, 2000)
    codes, ymask, _ = _record(L, T + U + n, C)
    w = _model(T, U, attention, U, C)
    rng = np.random.default_rng(n)
    starts = rng.integers(0, L - T + 1, size=n)
    starts[0] = L - T                          # windows at both ends of the record
    if n > 1:
        starts[1] = 0
    dropout = {"nodrop": 0.0, "holes": 0.5}.get(masks, 0.25)
    keep = (rng.random((n, 2, 5)) < 1 - dropout).astype(np.uint8)
    if masks in ("keep", "nodrop"):
        keep[:] = 1
    if masks == "holes":
        keep[1, 0] = 0
        keep[2, 1] = 0
        starts[3] = 1000
        codes[1000:1000 + T] = 4
    tr = _trainer(gpu_ctx, w, codes, ymask, dropout=dropout)
    loss = tr.step(starts, keep)
    grads = tr.grads()
    tr.close()
    _check_step(loss, grads, _w64(w), codes, ymask, starts, keep, dropout, T)


def test_clipped_loss_matches_the_oracle(gpu_ctx):
    """Keras clips the normalised probability of a labelled class to [1e-7, 1 - 1e-7] and passes no gradient
    through a clipped entry.  Large FF weights spread the logits so that labelled classes sit far below the clip
    range, far above it, and at moderate probabilities (some small but unclipped, about 1e-5); the labels are chosen
    from the float64 probabilities.  No labelled probability is within a factor of 10 of either clip boundary, where
    float32 and float64 could legitimately fall on different sides.

    One known difference needs no fix: 1.0f - 1e-7f rounds to 1 - 1.19e-7, while the oracle clamps at 1 - 1e-7.
    A labelled entry clipped at the top adds -log(1 - 1.19e-7) instead of -log(1 - 1e-7) to the sum, about 2e-8
    per position, far below the bounds."""
    T, U, C, n, dropout = 64, 8, 3, 6, 0.25
    w = dgmodel.random_weights(T, U, attention=True, n_classes=C, seed=21).scaled(2.0)
    rng = np.random.default_rng(21)
    w.ff_kernel = (rng.normal(size=w.ff_kernel.shape) * 30).astype(np.float32)
    w.ff_bias = np.linspace(10, -10, C).astype(np.float32)
    L = n * T
    codes = rng.integers(0, 4, size=L).astype(np.uint8)
    starts = np.arange(n) * T                 # the windows tile the record: every position in one window
    keep = (rng.random((n, 2, 5)) < 1 - dropout).astype(np.uint8)
    w64 = _w64(w)
    _, _, probs = train_oracle.train_loss_and_grads(w64, codes, np.zeros(L, np.uint8), starts, keep, dropout, T)
    p = (probs / probs.sum(-1, keepdims=True)).reshape(L, C)
    ymask = np.zeros(L, np.uint8)
    for i, q in enumerate(p):
        top = int(np.argmax(q))
        low = [c for c in range(C) if q[c] < (1e-8 if i % 2 else 1e-10)]
        mid = [c for c in range(C) if 1e-6 < q[c] < 1 - 1e-6]
        if 1 - q[top] < 1e-8 and i % 4 != 3:
            ymask[i] = 1 << top
        elif i % 3 == 0 and low:
            ymask[i] = 1 << max(low, key=lambda c: q[c])
        elif mid:
            ymask[i] = 1 << mid[i % len(mid)]
            if i % 5 == 0 and low:
                ymask[i] |= 1 << low[0]
    labelled = p[((ymask[:, None] >> np.arange(C)) & 1).astype(bool)]
    assert (labelled <= 1e-10).mean() >= 0.05 and (1 - labelled < 1e-8).mean() >= 0.05
    assert ((labelled > 1e-6) & (labelled < 1e-4)).sum() >= 5
    assert not ((labelled > 1e-8) & (labelled < 1e-6)).any()
    assert not ((1 - labelled > 1e-8) & (1 - labelled < 1e-6)).any()
    tr = _trainer(gpu_ctx, w, codes, ymask, dropout=dropout)
    loss = tr.step(starts, keep)
    grads = tr.grads()
    tr.close()
    _check_step(loss, grads, w64, codes, ymask, starts, keep, dropout, T)


def test_eval_probabilities_are_the_inference_model(gpu_ctx):
    T, U, L = 120, 32, 3000
    codes, ymask, _ = _record(L, 1)
    w = _model(T, U, True, 3)
    starts = np.array([0, 5, 1234, L - T])
    tr = _trainer(gpu_ctx, w, codes, ymask)
    loss, probs = tr.evaluate(1, starts, probs=True)
    tr.close()
    batch = np.eye(5, dtype=np.float32)[codes[starts[:, None] + np.arange(T)]]
    ref = dgpred.forward_windows(w, batch)
    assert np.abs(probs - ref).max() <= 1e-6
    assert np.isfinite(loss) and loss > 0


@pytest.mark.parametrize("C", [2, 5])
@pytest.mark.parametrize("attention", [True, False])
@pytest.mark.parametrize("U", [1, 33, 64])
def test_trained_model_evaluates_as_the_inference_model(gpu_ctx, U, attention, C):
    """After a few steps the trainer's evaluation and prediction's forward compute the same model."""
    T, L, n = 40, 1500, 8
    codes, ymask, _ = _record(L, 50 + U, C)
    tr = _trainer(gpu_ctx, _model(T, U, attention, 51, C), codes, ymask, dropout=0.25, learning_rate=3e-3)
    rng = np.random.default_rng(52)
    for _ in range(3):
        tr.step(rng.integers(0, L - T + 1, size=n), (rng.random((n, 2, 5)) < 0.75).astype(np.uint8))
    starts = np.array([0, 1, 777, L - T])
    _, probs = tr.evaluate(1, starts, probs=True)
    model = tr.model()
    tr.close()
    ref = dgpred.forward_windows(model, np.eye(5, dtype=np.float32)[codes[starts[:, None] + np.arange(T)]])
    assert np.abs(probs - ref).max() <= 1e-6


def _check_eval(loss, probs, w64, codes, ymask, starts, T):
    """An evaluation (no dropout) against the float64 oracle: loss within max(1e-5, 8 e32) relative, probabilities
    within max(1e-5, 8 e32) absolute."""
    keep = np.ones((len(starts), 2, 5), np.uint8)
    loss_o, grads_o, probs_o = train_oracle.train_loss_and_grads(w64, codes, ymask, starts, keep, 0.0, T)
    e = _e32(w64, codes, ymask, starts, keep, 0.0, T, loss_o, grads_o, probs_o)
    assert abs(loss - loss_o) <= max(1e-5, 8 * e["loss"]) * loss_o, (loss, loss_o)
    if probs is not None:
        assert np.abs(probs - probs_o).max() <= max(1e-5, 8 * e["probs"])


def test_evaluation_reads_the_validation_record_and_the_current_weights(gpu_ctx):
    T, U = 50, 16
    codes0, ymask0, _ = _record(3000, 31)
    codes1, ymask1, _ = _record(700, 32)           # shorter than the training record, and different
    w = _model(T, U, True, 33)
    tr = dgtrain.Trainer(w, dgmodel.Options(dropout=0.25), gpu_ctx)
    tr.set_data(0, codes0, ymask0)
    tr.set_data(1, codes1, ymask1)
    starts = np.array([0, 17, 333, 700 - T])
    loss, probs = tr.evaluate(1, starts, probs=True)
    _check_eval(loss, probs, _w64(w), codes1, ymask1, starts, T)
    with pytest.raises(_lib.DeepgrpError, match="outside") as e:   # record 0 would be long enough
        tr.evaluate(1, np.array([0, 700 - T + 1]))
    assert e.value.code == _lib.E_ARG
    assert np.isfinite(tr.evaluate(0, np.array([0, 700 - T + 1])))
    rng = np.random.default_rng(34)
    for _ in range(3):
        tr.step(rng.integers(0, 3000 - T + 1, size=8), (rng.random((8, 2, 5)) < 0.75).astype(np.uint8))
    w3 = tr.weights()
    _check_eval(tr.evaluate(1, starts), None, _w64(w3), codes1, ymask1, starts, T)
    tr.close()


def test_evaluation_in_several_passes(gpu_ctx):
    """2 * 1024 + 37 windows run as three forward passes; every window is computed on its own, so the probabilities
    are those of three calls on the slices, bit for bit."""
    T, U, L = 8, 4, 4000
    n = 2 * 1024 + 37
    codes, ymask, _ = _record(L, 35)
    w = _model(T, U, True, 36)
    tr = _trainer(gpu_ctx, w, codes, ymask)
    starts = np.random.default_rng(37).integers(0, L - T + 1, size=n)
    loss, probs = tr.evaluate(1, starts, probs=True)
    sliced = [tr.evaluate(1, starts[a:b], probs=True) for a, b in ((0, 1024), (1024, 2048), (2048, n))]
    tr.close()
    assert np.array_equal(probs, np.concatenate([p for _, p in sliced]))
    assert abs(loss - (1024 * sliced[0][0] + 1024 * sliced[1][0] + 37 * sliced[2][0]) / n) <= 1e-6 * loss
    _check_eval(loss, None, _w64(w), codes, ymask, starts, T)


def test_step_loss_is_the_evaluation_loss(gpu_ctx):
    """Without dropout a step's forward is the evaluation's: the same loss, bit for bit."""
    T, U, L, n = 60, 16, 2000, 32
    codes, ymask, _ = _record(L, 38)
    tr = _trainer(gpu_ctx, _model(T, U, True, 39), codes, ymask, dropout=0.0)
    starts = np.random.default_rng(40).integers(0, L - T + 1, size=n)
    before = tr.evaluate(0, starts)
    assert tr.step(starts, np.ones((n, 2, 5), np.uint8)) == before
    tr.close()


def test_replacing_a_record(gpu_ctx):
    """A shorter record replaces the training record (its device buffers only grow, so stale bytes remain past the
    new end); a refused upload leaves the previous record in place."""
    T, U = 40, 16
    codes, ymask, _ = _record(3000, 41)
    tr = _trainer(gpu_ctx, _model(T, U, True, 42), codes, ymask, dropout=0.25)
    rng = np.random.default_rng(43)
    tr.step(np.array([0, 3000 - T]), np.ones((2, 2, 5), np.uint8))
    codes2, ymask2, _ = _record(900, 44)
    tr.set_data(0, codes2, ymask2)
    with pytest.raises(_lib.DeepgrpError, match="outside") as e:
        tr.step(np.array([3000 - T]), np.ones((1, 2, 5), np.uint8))
    assert e.value.code == _lib.E_ARG
    for _ in range(2):
        starts = rng.integers(0, 900 - T + 1, size=6)
        starts[0] = 900 - T
        keep = (rng.random((6, 2, 5)) < 0.75).astype(np.uint8)
        w = tr.weights()
        loss = tr.step(starts, keep)
        _check_step(loss, tr.grads(), _w64(w), codes2, ymask2, starts, keep, 0.25, T)
    starts = np.array([0, 123, 900 - T])
    before = [tr.evaluate(0, starts), tr.evaluate(1, starts)]
    bad_code, bad_label = codes2.copy(), ymask2.copy()
    bad_code[400] = 5
    bad_label[400] = 1 << 5
    for which in (0, 1):
        with pytest.raises(_lib.DeepgrpError, match="base code") as e:
            tr.set_data(which, bad_code, ymask2)
        assert e.value.code == _lib.E_ARG
        with pytest.raises(_lib.DeepgrpError, match="names a class") as e:
            tr.set_data(which, codes2, bad_label)
        assert e.value.code == _lib.E_ARG
    assert [tr.evaluate(0, starts), tr.evaluate(1, starts)] == before
    tr.close()


def _ulp32(a):
    return np.spacing(np.abs(a).astype(np.float32)).astype(np.float64)


@pytest.mark.parametrize("optimizer,momentum,rho,epsilon", [
    ("RMSprop", 0.9, 0.8, 1e-6),
    ("RMSprop", 0.0, 0.9, 1e-10),
    ("Adam", 0.0, 0.9, 1e-7),
])
def test_optimizer_state_over_forty_steps(gpu_ctx, optimizer, momentum, rho, epsilon):
    """Teacher-forced: every update is checked from the GPU's own previous weights and gradients, with the oracle's
    float64 state fed by those gradients alone.  Errors of the weights cannot compound, so the bound stays tight
    over all steps and pins the state carry and (Adam) the step counter; evaluations between steps must not advance
    it.

    Bound: 2 ulp32 of the weight, 1e-5 of the update, and the float32 rounding that the GPU's first-moment state
    (RMSprop mom, Adam m) carries from step to step.  Each step rounds that state and the error decays by momentum
    (beta1), so `carry` sums the ulp32 of the state with that decay.  It matters only where the state nearly cancels,
    leaving an update much smaller than the state it came from."""
    T, U, L, n, steps, lr = 30, 8, 2000, 8, 40, 2e-3
    codes, ymask, y = _record(L, 45)
    opts = dict(vecsize=T, batch_size=n, dropout=0.25, optimizer=optimizer, learning_rate=lr, rho=rho,
                momentum=momentum, epsilon=epsilon)
    tr = _trainer(gpu_ctx, _model(T, U, True, 46), codes, ymask, **opts)
    sampler = dgtrain.BatchSampler(y, dgmodel.Options(**opts))
    rng = np.random.default_rng(47)
    state, carry = {k: {} for k in NAMES}, {k: 0.0 for k in NAMES}
    prev = tr.weights()
    for k in range(1, steps + 1):
        d = sampler.draw(rng)
        tr.step(d.starts, d.keep)
        g, cur = tr.grads(), tr.weights()
        for name in NAMES:
            if prev[name] is None:
                continue
            ref, state[name] = train_oracle.optimizer_step(optimizer, prev[name], g[name], state[name], k, lr, rho,
                                                           momentum, epsilon)
            if optimizer == "Adam":
                carry[name] = 0.9 * carry[name] + _ulp32(state[name]["m"])
                lr_t = lr * np.sqrt(1 - 0.999 ** k) / (1 - 0.9 ** k)
                state_err = lr_t * carry[name] / (np.sqrt(state[name]["v"]) + epsilon)
            elif momentum > 0:
                carry[name] = momentum * carry[name] + _ulp32(state[name]["mom"])
                state_err = carry[name]
            else:
                state_err = 0.0
            bound = 2 * _ulp32(ref) + 1e-5 * np.abs(ref - prev[name]) + state_err
            err = np.abs(cur[name] - ref)
            assert (err <= bound).all(), (k, name, float((err / bound).max()))
        if optimizer == "Adam" and k % 10 == 5:
            tr.evaluate(1, d.starts)
            tr.evaluate(0, d.starts, probs=True)
        prev = cur
    tr.close()


@pytest.mark.parametrize("optimizer,momentum", [("RMSprop", 0.9), ("RMSprop", 0.0), ("Adam", 0.9)])
def test_zero_learning_rate_keeps_the_weights(gpu_ctx, optimizer, momentum):
    T, U, L, n = 30, 8, 2000, 8
    codes, ymask, _ = _record(L, 48)
    w = _model(T, U, True, 49)
    tr = _trainer(gpu_ctx, w, codes, ymask, optimizer=optimizer, momentum=momentum, learning_rate=0.0,
                  dropout=0.25)
    rng = np.random.default_rng(50)
    for _ in range(4):
        tr.step(rng.integers(0, L - T + 1, size=n), (rng.random((n, 2, 5)) < 0.75).astype(np.uint8))
    got = tr.weights()
    tr.close()
    for name in NAMES:
        assert np.array_equal(got[name], getattr(w, name)), name


@pytest.mark.parametrize("optimizer,momentum", [("RMSprop", 0.9), ("RMSprop", 0.0), ("Adam", 0.9)])
def test_one_optimizer_step_matches_the_oracle_rule(gpu_ctx, optimizer, momentum):
    T, U, L = 60, 16, 2000
    codes, ymask, _ = _record(L, 2)
    w = _model(T, U, True, 5)
    opts = dict(optimizer=optimizer, momentum=momentum, learning_rate=2e-3, rho=0.8, epsilon=1e-7)
    tr = _trainer(gpu_ctx, w, codes, ymask, **opts)
    rng = np.random.default_rng(3)
    tr.step(rng.integers(0, L - T + 1, size=16), (rng.random((16, 2, 5)) < 0.75).astype(np.uint8))
    g, w1 = tr.grads(), tr.weights()
    tr.close()
    for name in NAMES:
        ref, _ = train_oracle.optimizer_step(optimizer, getattr(w, name), g[name], {}, 1, 2e-3, 0.8, momentum, 1e-7)
        assert _rel(w1[name], ref) <= 1e-6, (name, _rel(w1[name], ref))


def test_twenty_steps_follow_the_oracle(gpu_ctx):
    """20 RMSprop steps (the defaults: lr 1e-3, rho 0.9, momentum 0.9, eps 1e-10) on the same batches and masks:
    the GPU's fp32 weights against the oracle's float64 trajectory."""
    T, U, L, n, steps = 40, 16, 2000, 8, 20
    codes, ymask, y = _record(L, 4)
    w = _model(T, U, True, 6)
    options = dgmodel.Options(vecsize=T, batch_size=n, dropout=0.25)
    tr = _trainer(gpu_ctx, w, codes, ymask, vecsize=T, batch_size=n, dropout=0.25)
    sampler = dgtrain.BatchSampler(y, options)
    rng = np.random.default_rng(7)
    w64, state = _w64(w), {k: {} for k in NAMES}
    for step in range(1, steps + 1):
        d = sampler.draw(rng)
        tr.step(d.starts, d.keep)
        _, g, _ = train_oracle.train_loss_and_grads(w64, codes, ymask, d.starts, d.keep, 0.25, T)
        for name in g:
            w64[name], state[name] = train_oracle.optimizer_step("RMSprop", w64[name], g[name], state[name], step,
                                                           1e-3, 0.9, 0.9, 1e-10)
    got = tr.weights()
    tr.close()
    for name in g:
        assert _rel(got[name], w64[name]) <= 1e-3, (name, _rel(got[name], w64[name]))


def test_training_is_bit_reproducible(gpu_ctx):
    T, U, L, n = 100, 32, 5000, 64
    codes, ymask, _ = _record(L, 5)
    results = []
    for _ in range(2):
        tr = _trainer(gpu_ctx, _model(T, U, True, 7), codes, ymask, vecsize=T, batch_size=n)
        rng = np.random.default_rng(9)
        losses = [tr.step(rng.integers(0, L - T + 1, size=n), (rng.random((n, 2, 5)) < 0.75).astype(np.uint8))
                  for _ in range(10)]
        results.append((losses, tr.weights()))
        tr.close()
    assert results[0][0] == results[1][0]
    for name in NAMES:
        assert np.array_equal(results[0][1][name], results[1][1][name]), name


# ---- a model that learns -----------------------------------------------------------------------------------------

_UNIT = np.array([0, 2, 3, 1, 1, 0, 3], np.int64)      # class 1: tandem copies of AGTCCAT


def _planted(length, seed, element):
    """Seeded random DNA with one planted repeat per 1 kb slot, alternating class 1 (a tandem array of _UNIT,
    120-280 bp) and class 2 (a copy of `element` with 10 % point mutations).  Returns (codes, labels [3, L])."""
    rng = np.random.default_rng(seed)
    seq = rng.integers(0, 4, size=length)
    y = np.zeros((3, length), np.int8)
    for k, slot in enumerate(range(0, length - 1000, 1000)):
        if k % 2 == 0:
            ln = int(rng.integers(120, 281))
            ins = np.resize(_UNIT, ln)
            cls = 1
        else:
            ins = element.copy()
            mut = rng.random(ins.size) < 0.1
            ins[mut] = rng.integers(0, 4, size=int(mut.sum()))
            cls = 2
        a = slot + int(rng.integers(50, 1000 - ins.size - 50))
        seq[a:a + ins.size] = ins
        y[cls, a:a + ins.size] = 1
    y[0, ~y[1:].any(axis=0)] = 1
    return seq.astype(np.uint8), y


def _write_bed(path, chrom_labels):
    with open(path, "w") as fh:
        for chrom, y in chrom_labels:
            for cls in (1, 2):
                edges = np.flatnonzero(np.diff(np.concatenate([[0], y[cls], [0]])))
                for a, b in zip(edges[::2], edges[1::2]):
                    fh.write("%s\t%d\t%d\t%d\n" % (chrom, a, b, cls))


def _recall(rows_tsv, y):
    pred = np.zeros(y.shape[1], np.int64)
    for line in open(rows_tsv):
        _, _, s, e, lab = line.rstrip("\n").split("\t")
        pred[int(s):int(e)] = int(lab)
    return [float((pred[y[c] == 1] == c).mean()) for c in (1, 2)]


def test_it_learns_planted_repeats(gpu_ctx, tmp_path):
    """Train (T=100, U=16, attention) on 60 kb with 30 tandem arrays and 30 mutated copies of one 300-bp element,
    validate on 30 kb, then `deepgrp predict` a held-out 30 kb record with the saved best.hdf5.

    First observed run (B200, 60 epochs of 25 steps, 0.9 s): validation loss 0.9045 after the first epoch, best 0.1990
    (0.22 of it); held-out recall 0.972 (tandem) and 0.814 (element).  The thresholds keep a margin of about 0.12-0.16
    below those recalls, and the loss criterion (below half) a factor of 2.3."""
    element = np.random.default_rng(99).integers(0, 4, size=300)
    codes_t, y_t = _planted(60_000, 1, element)
    codes_v, y_v = _planted(30_000, 2, element)
    codes_h, y_h = _planted(30_000, 3, element)
    options = dgmodel.Options(vecsize=100, units=16, attention=True, batch_size=64, n_batches=25, n_epochs=60,
                              early_stopping_th=10, repeats_to_search=[1, 2])
    model = dgmodel.create_model(options)
    data = (dgprep.Data(np.eye(5, dtype=np.int8)[codes_t].T, y_t), dgprep.Data(np.eye(5, dtype=np.int8)[codes_v].T, y_v))
    logdir = str(tmp_path / "logs")
    history = dgtrain.training(data, options, model, logdir, seed=0)
    val = [h[2] for h in history]
    print("epochs %d, val loss first %.4f best %.4f" % (len(val), val[0], min(val)))
    assert min(val) < 0.5 * val[0]
    fasta = tmp_path / "held.fa"
    fasta.write_text(">held\n" + "".join("ACGT"[c] for c in codes_h) + "\n")
    out = tmp_path / "rows.tsv"
    cli.CommandLineParser().parse_args(["predict", os.path.join(logdir, "best.hdf5"), str(fasta), "--output",
                                        str(out)]).run()
    recall = _recall(str(out), y_h)
    print("held-out recall: tandem %.3f, element %.3f" % tuple(recall))
    assert recall[0] >= 0.85 and recall[1] >= 0.65, recall


def test_cli_train_then_predict(gpu_ctx, tmp_path):
    element = np.random.default_rng(98).integers(0, 4, size=300)
    codes_t, y_t = _planted(20_000, 4, element)
    codes_v, y_v = _planted(10_000, 5, element)
    train, valid = str(tmp_path / "chrA.fa.gz.npz"), str(tmp_path / "chrB.fa.gz.npz")
    np.savez_compressed(train, fwd=np.eye(5, dtype=np.int8)[codes_t].T, hash=np.array(["a"]))
    np.savez_compressed(valid, fwd=np.eye(5, dtype=np.int8)[codes_v].T, hash=np.array(["b"]))
    bed = str(tmp_path / "rm.bed")
    _write_bed(bed, [("chrA", y_t), ("chrB", y_v)])
    params = tmp_path / "params.toml"
    params.write_text("vecsize = 100\nunits = 16\nattention = true\nbatch_size = 64\nn_batches = 25\n"
                      "n_epochs = 12\nearly_stopping_th = 12\nrepeats_to_search = [1, 2]\nlearning_rate = 0.003\n")
    logdir, modelfile = str(tmp_path / "D"), str(tmp_path / "m.hdf5")
    cli.CommandLineParser().parse_args(["train", str(params), train, valid, bed, "--logdir", logdir,
                                        "--modelfile", modelfile]).run()
    assert os.path.exists(os.path.join(logdir, "best.hdf5"))
    assert len(open(os.path.join(logdir, "history.tsv")).read().splitlines()) == 13
    codes_x, _ = _planted(6_000, 6, element)
    fasta = tmp_path / "x.fa"
    fasta.write_text(">x\n" + "".join("ACGT"[c] for c in codes_x) + "\n")
    out = tmp_path / "rows.tsv"
    cli.CommandLineParser().parse_args(["predict", modelfile, str(fasta), "--output", str(out)]).run()
    rows = [line.split("\t") for line in out.read_text().splitlines()]
    assert rows and all(len(r) == 5 and r[1] == "x" and int(r[4]) in (1, 2) for r in rows)
    # predict_complete restores D/best.hdf5
    options = dgmodel.Options(vecsize=100, batch_size=64)
    data = dgprep.Data(np.eye(5, dtype=np.int8)[codes_x].T, np.zeros((3, codes_x.size), np.int8))
    got = dgpred.predict_complete(50, options, logdir, data)
    best = dgmodel.load_model(os.path.join(logdir, "best.hdf5"))
    ref = dgpred.softmax(dgpred.predict(best, dgpred.fetch_validation_batch(data.fwd, 50, 64, 100),
                                        (codes_x.size, 3), 50))
    assert np.array_equal(got, ref)


# ---- refusals ----------------------------------------------------------------------------------------------------

def test_refusals(gpu_ctx, tmp_path):
    codes, ymask, _ = _record(500, 6)
    for C, code in ((1, _lib.E_ARG), (6, _lib.E_UNSUPPORTED)):
        with pytest.raises(_lib.DeepgrpError, match="n_classes") as e:
            dgtrain.Trainer(dgmodel.random_weights(50, 8, n_classes=C), dgmodel.Options(), gpu_ctx)
        assert e.value.code == code
    assert "prediction" in str(e.value)
    for C in (2, 5):
        dgtrain.Trainer(dgmodel.random_weights(50, 8, n_classes=C), dgmodel.Options(), gpu_ctx).close()
    t_max = _max_vecsize(gpu_ctx, 64, 5, True)
    with pytest.raises(_lib.DeepgrpError, match="shared memory") as e:
        dgtrain.Trainer(dgmodel.random_weights(t_max + 1, 64, n_classes=5), dgmodel.Options(), gpu_ctx)
    assert e.value.code == _lib.E_UNSUPPORTED
    # six classes (five repeat types): refused before the first epoch, so no model prediction cannot run is written
    options = dgmodel.Options(vecsize=50, units=8, batch_size=4, n_batches=2, n_epochs=1,
                              repeats_to_search=[1, 2, 3, 4, 5])
    _, _, y6 = _record(500, 7, 6)
    data = dgprep.Data(np.eye(5, dtype=np.int8)[codes].T, y6)
    logdir = str(tmp_path / "logs")
    with pytest.raises(_lib.DeepgrpError, match="prediction") as e:
        dgtrain.training((data, data), options, dgmodel.create_model(options), logdir)
    assert e.value.code == _lib.E_UNSUPPORTED
    assert not os.path.exists(os.path.join(logdir, "history.tsv"))
    with pytest.raises(_lib.DeepgrpError, match="LSTM") as e:
        dgtrain.Trainer(dgmodel.random_weights(50, 8, rnn="LSTM"), dgmodel.Options(), gpu_ctx)
    assert e.value.code == _lib.E_UNSUPPORTED
    with pytest.raises(_lib.DeepgrpError, match="units <= 64") as e:
        dgtrain.Trainer(dgmodel.random_weights(50, 65), dgmodel.Options(), gpu_ctx)
    assert e.value.code == _lib.E_UNSUPPORTED
    with pytest.raises(ValueError, match="optimizer"):
        dgtrain.Trainer(dgmodel.random_weights(50, 8), dgmodel.Options(optimizer="SGD"), gpu_ctx)
    tr = dgtrain.Trainer(dgmodel.random_weights(50, 8), dgmodel.Options(), gpu_ctx)
    keep = np.ones((1, 2, 5), np.uint8)
    with pytest.raises(_lib.DeepgrpError, match="no training data set") as e:
        tr.step(np.array([0]), keep)
    assert e.value.code == _lib.E_ARG
    with pytest.raises(_lib.DeepgrpError, match="shorter than vecsize") as e:
        tr.set_data(0, codes[:49], ymask[:49])
    assert e.value.code == _lib.E_ARG
    tr.set_data(0, codes, ymask)
    for bad in (-1, 451):
        with pytest.raises(_lib.DeepgrpError, match="outside") as e:
            tr.step(np.array([0, bad]), np.ones((2, 2, 5), np.uint8))
        assert e.value.code == _lib.E_ARG
    with pytest.raises(_lib.DeepgrpError, match="at least 1") as e:
        tr.step(np.zeros(0, np.int64), np.ones((0, 2, 5), np.uint8))
    assert e.value.code == _lib.E_ARG
    assert np.isfinite(tr.step(np.array([0, 450]), np.ones((2, 2, 5), np.uint8)))
    tr.close()
