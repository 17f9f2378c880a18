"""Training on the GPU (csrc/train.cu through dgrp_train_*): gradients and updates against the float64 oracle,
the trainer's forward against inference, determinism, a model that learns planted repeats, the CLI end to end and
the refusals."""
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


@pytest.mark.parametrize("T,U,attention,n,masks,C", [
    (150, 32, True, 3, "random", 5),
    (342, 60, True, 256, "random", 5),
    (40, 16, False, 1, "keep", 8),
    (40, 16, False, 3, "random", 5),
    (7, 1, True, 3, "random", 5),
    (64, 64, True, 3, "keep", 5),
    (150, 32, True, 256, "keep", 5),
])
def test_gradients_match_the_float64_oracle(gpu_ctx, T, U, attention, n, masks, C):
    L = max(4 * T, 2000)
    codes, ymask, _ = _record(L, T + U + n, C)
    w = _model(T, U, attention, U, C)
    rng = np.random.default_rng(n)
    starts = rng.integers(0, L - T + 1, size=n)
    starts[0] = L - T                          # windows at both ends of the record
    if n > 1:
        starts[1] = 0
    dropout = 0.25
    keep = (rng.random((n, 2, 5)) < 0.75).astype(np.uint8) if masks == "random" else np.ones((n, 2, 5), np.uint8)
    tr = _trainer(gpu_ctx, w, codes, ymask, dropout=dropout)
    loss = tr.step(starts, keep)
    grads = tr.grads()
    tr.close()
    loss_o, grads_o, _ = train_oracle.train_loss_and_grads(_w64(w), codes, ymask, starts, keep, dropout, T)
    assert abs(loss - loss_o) <= 1e-5 * abs(loss_o)
    assert set(grads_o) == {k for k in NAMES if grads[k] is not None}
    for name, g in grads_o.items():
        # bias rows separately: row 0 (input) and row 1 (recurrent) come from different sums
        parts = [(name, grads[name], g)] if name != "bias" else [("bias0", grads[name][0], g[0]),
                                                                  ("bias1", grads[name][1], g[1])]
        for label, got, ref in parts:
            assert _rel(got, ref) <= 1e-4, (label, _rel(got, ref))


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

def test_refusals(gpu_ctx):
    codes, ymask, _ = _record(500, 6)
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
