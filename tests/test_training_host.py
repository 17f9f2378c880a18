"""Training without a GPU: the float64 oracle against the model and against finite differences, the window sampler,
and the `deepgrp train` wiring with `training` replaced by a stand-in."""
import argparse

import numpy as np
import pytest

from deepgrp_b200 import __main__ as cli
from deepgrp_b200 import model as dgmodel
from deepgrp_b200 import training as dgtrain
from oracle import train_oracle


def _record(length, seed, n_classes=5):
    """Random base codes (a few N) and a multi-hot label mask with overlapping annotations."""
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, 4, size=length).astype(np.uint8)
    codes[rng.random(length) < 0.02] = 4
    y = np.zeros((n_classes, length), np.int8)
    for c in range(1, n_classes):
        for _ in range(3):
            a = int(rng.integers(0, length - 10))
            y[c, a:a + int(rng.integers(5, 40))] = 1
    y[0, ~y[1:].any(axis=0)] = 1
    return codes, dgtrain.labels_to_mask(y), y


def _weights(T, U, attention, seed, C=5, scale=1.0):
    w = dgmodel.random_weights(T, U, attention=attention, n_classes=C, seed=seed)
    d = {k: v * scale for k, v in w.as_dict().items()}
    rng = np.random.default_rng(seed + 100)
    d["bias"] = (rng.normal(size=d["bias"].shape) * 0.1).astype(np.float32)   # non-zero biases reach every term
    d["ff_bias"] = (rng.normal(size=d["ff_bias"].shape) * 0.1).astype(np.float32)
    return d


@pytest.mark.parametrize("attention", [True, False])
def test_oracle_training_forward_is_the_model(oracle, attention):
    T, U = 30, 8
    codes, ymask, _ = _record(200, 1)
    w = _weights(T, U, attention, 2, scale=2.0)
    starts = np.array([0, 17, 170, 93])
    keep = np.ones((starts.size, 2, 5), np.uint8)
    _, _, probs = train_oracle.train_loss_and_grads(w, codes, ymask, starts, keep, 0.0, T)
    batch = np.eye(5)[codes[starts[:, None] + np.arange(T)]]
    ref = oracle.model_forward(batch, {k: np.float64(v) for k, v in w.items()}, dtype=np.float64)
    assert np.abs(probs - ref).max() <= 1e-12


@pytest.mark.parametrize("attention", [True, False])
def test_oracle_gradients_match_finite_differences(attention):
    """Central differences of the float64 loss pin the oracle's autograd gradients to the stated math."""
    T, U = 5, 3
    codes, ymask, _ = _record(40, 3)
    w = {k: np.float64(v) for k, v in _weights(T, U, attention, 4, scale=1.5).items()}
    starts = np.array([0, 9, 35])
    keep = (np.random.default_rng(5).random((3, 2, 5)) < 0.7).astype(np.uint8)
    dropout = 0.3
    _, grads, _ = train_oracle.train_loss_and_grads(w, codes, ymask, starts, keep, dropout, T)

    def loss_at(name, i, delta):
        v = {k: a.copy() for k, a in w.items()}
        v[name].reshape(-1)[i] += delta
        return train_oracle.train_forward(v, codes, ymask, starts, keep, dropout, T)[0].item()
    h = 1e-6
    for name, g in grads.items():
        fd = np.array([(loss_at(name, i, h) - loss_at(name, i, -h)) / (2 * h) for i in range(g.size)])
        err = np.linalg.norm(fd - g.reshape(-1)) / max(np.linalg.norm(g), 1e-12)
        assert err <= 1e-6, (name, err)
    assert set(grads) == {k for k, v in w.items() if v is not None}


@pytest.mark.parametrize("attention", [True, False])
def test_oracle_float32_is_float64_to_rounding_noise(attention):
    """The float32 run of the oracle (the GPU tests' measure of a shape's rounding noise) is the same math: it agrees
    with float64 to float32 noise, and asking for float64 explicitly changes no bit of the default result."""
    import torch
    T, U = 12, 6
    codes, ymask, _ = _record(120, 12)
    w = _weights(T, U, attention, 13, scale=2.0)
    starts = np.array([0, 31, 108])
    keep = (np.random.default_rng(14).random((3, 2, 5)) < 0.75).astype(np.uint8)
    loss, grads, probs = train_oracle.train_loss_and_grads(w, codes, ymask, starts, keep, 0.25, T)
    loss64, grads64, probs64 = train_oracle.train_loss_and_grads(w, codes, ymask, starts, keep, 0.25, T,
                                                                  dtype=torch.float64)
    assert loss == loss64 and np.array_equal(probs, probs64) and probs.dtype == np.float64
    assert all(np.array_equal(grads[k], grads64[k]) and grads[k].dtype == np.float64 for k in grads)
    loss32, grads32, probs32 = train_oracle.train_loss_and_grads(w, codes, ymask, starts, keep, 0.25, T,
                                                                  dtype=torch.float32)
    assert probs32.dtype == np.float32 and set(grads32) == set(grads)
    assert abs(loss32 - loss) <= 1e-6 * loss
    assert np.abs(probs32 - probs).max() <= 1e-6
    for k, g in grads.items():
        assert grads32[k].dtype == np.float32
        err = np.linalg.norm(grads32[k] - g) / np.linalg.norm(g)
        assert 0 < err <= 1e-4, (k, err)      # 0 would mean the float32 path did not run in float32


def test_optimizer_step_rules():
    w, g = np.array([1.0, -2.0]), np.array([0.5, -0.25])
    new, st = train_oracle.optimizer_step("RMSprop", w, g, {}, 1, 0.1, 0.9, 0.5, 1e-10)
    ms = 0.1 * g * g
    assert np.allclose(st["ms"], ms) and np.allclose(new, w - 0.1 * g / np.sqrt(ms + 1e-10))
    new, _ = train_oracle.optimizer_step("RMSprop", w, g, {}, 1, 0.1, 0.9, 0.0, 1e-10)
    assert np.allclose(new, w - 0.1 * g / (np.sqrt(ms) + 1e-10))
    new, st = train_oracle.optimizer_step("Adam", w, g, {}, 1, 0.1, epsilon=1e-7)
    assert np.allclose(new, w - 0.1 * np.sign(g), atol=1e-5)      # the first Adam step is lr * sign(g)
    with pytest.raises(ValueError):
        train_oracle.optimizer_step("SGD", w, g, {}, 1)


# ---- sampler ----------------------------------------------------------------------------------------------------

def _sampler_options(**kw):
    base = dict(vecsize=50, batch_size=4000, repeat_probability=0.3, dropout=0.25, repeats_to_search=[1, 2, 3, 4])
    base.update(kw)
    return dgmodel.Options(**base)


def test_sampler_is_seeded_and_in_range():
    _, _, y = _record(3000, 7)
    s = dgtrain.BatchSampler(y, _sampler_options())
    a, b = s.draw(np.random.default_rng(11)), s.draw(np.random.default_rng(11))
    assert all(np.array_equal(x, z) for x, z in zip(a, b))
    c = s.draw(np.random.default_rng(12))
    assert not np.array_equal(a.starts, c.starts)
    assert a.starts.dtype == np.int64 and a.keep.shape == (4000, 2, 5) and a.keep.dtype == np.uint8
    assert a.starts.min() >= 0 and a.starts.max() <= 3000 - 50


def test_sampler_repeat_windows_contain_their_class():
    _, _, y = _record(3000, 8)
    y[3] = 0                                  # a searched class that does not occur is never drawn
    s = dgtrain.BatchSampler(y, _sampler_options())
    d = s.draw(np.random.default_rng(1))
    drawn = d.repeat_class >= 0
    assert set(np.unique(d.repeat_class[drawn])) == {1, 2, 4}
    for start, cls in zip(d.starts[drawn], d.repeat_class[drawn]):
        assert y[cls, start:start + 50].any()


def test_sampler_rates():
    _, _, y = _record(3000, 9)
    p, drop, n = 0.3, 0.25, 4000
    d = dgtrain.BatchSampler(y, _sampler_options(repeat_probability=p, dropout=drop)).draw(np.random.default_rng(2))
    frac = (d.repeat_class >= 0).mean()
    assert abs(frac - p) <= 3 * np.sqrt(p * (1 - p) / n)
    keep = d.keep.mean()
    assert abs(keep - (1 - drop)) <= 3 * np.sqrt(drop * (1 - drop) / d.keep.size)


def test_fetch_batch_shapes():
    codes, _, y = _record(500, 10)
    x = np.eye(5, dtype=np.int8)[codes].T
    xb, yb = next(dgtrain.fetch_batch(x, y, _sampler_options(batch_size=6), np.random.default_rng(0)))
    assert xb.shape == (6, 50, 5) and yb.shape == (6, 50, 5) and xb.dtype == yb.dtype == np.float32
    assert (xb.sum(axis=2) == 1).all()


def test_codes_and_masks():
    fwd = np.eye(5, dtype=np.int8)[[0, 4, 3, 2, 1]].T
    assert dgtrain.onehot_to_codes(fwd).tolist() == [0, 4, 3, 2, 1]
    fwd[:, 2] = 0
    with pytest.raises(ValueError):
        dgtrain.onehot_to_codes(fwd)
    y = np.array([[1, 0, 0], [0, 1, 1], [0, 0, 1]], np.int8)
    assert dgtrain.labels_to_mask(y).tolist() == [1, 2, 6]


def test_unknown_optimizer_is_a_value_error():
    with pytest.raises(ValueError, match="optimizer"):
        dgtrain.Trainer(dgmodel.random_weights(10, 4), dgmodel.Options(optimizer="SGD"))


# ---- CLI ---------------------------------------------------------------------------------------------------------

def _write_inputs(tmp_path, n=400):
    rng = np.random.default_rng(0)
    paths = []
    for name in ("chr7.fa.gz.npz", "chr9.fa.gz.npz"):
        fwd = np.eye(5, dtype=np.int8)[rng.integers(0, 4, size=n)].T.copy()
        fwd[:, :3] = 0
        fwd[4, :3] = 1                        # leading N columns are cut by drop_start_end_n
        path = str(tmp_path / name)
        np.savez_compressed(path, fwd=fwd, hash=np.array(["0"]))
        paths.append(path)
    bed = tmp_path / "rm.bed"
    bed.write_text("chr7 10 60 1\nchr7 50 90 2\nchr9 100 200 1\nchr1 0 300 2\n")
    params = tmp_path / "params.toml"
    params.write_text("vecsize = 40\nunits = 8\nattention = true\nbatch_size = 8\nn_epochs = 2\n")
    return paths, str(bed), str(params)


def test_cli_train_wiring(monkeypatch, tmp_path):
    (train, valid), bed, params = _write_inputs(tmp_path)
    seen = {}

    def fake_training(data, options, model, logdir, seed=0):
        seen.update(data=data, options=options, logdir=logdir)
        model.kernel = model.kernel * 2.0          # training leaves its result in the model
        return []
    monkeypatch.setattr(dgtrain, "training", fake_training)
    modelfile = str(tmp_path / "m.hdf5")
    cli.CommandLineParser().parse_args(["-b", "64", "-l", "33", "train", params, train, valid, bed, "--logdir",
                                        str(tmp_path / "logs"), "--modelfile", modelfile]).run()
    opt = seen["options"]
    assert (opt.vecsize, opt.units, opt.attention, opt.batch_size, opt.n_epochs) == (40, 8, True, 8, 2)   # TOML wins
    assert (opt.min_mss_len, opt.xdrop_len) == (33, 50)                      # the command line fills the rest
    tr, va = seen["data"]
    assert tr.fwd.shape == (5, 396) and tr.truelbl.shape == (5, 396)        # 3 N columns and the last column cut
    # chromosome rule: chr7.fa.gz.npz -> chr7 (chr9 for the validation file; chr1 rows belong to neither)
    assert tr.truelbl[1, 7:57].all() and tr.truelbl[2, 47:87].all() and not tr.truelbl[1, 57:].any()
    assert va.truelbl[1, 97:197].all() and not va.truelbl[2].any()
    assert seen["logdir"] == str(tmp_path / "logs")
    saved = dgmodel.load_model(modelfile)
    ref = dgmodel.create_model(opt)
    assert np.array_equal(saved.kernel, ref.kernel * 2.0)
    for name in ("recurrent_kernel", "bias", "att_scale", "ff_kernel", "ff_bias"):
        assert np.array_equal(getattr(saved, name), getattr(ref, name)), name
    assert saved.vecsize == 40


def test_cli_train_rejects_a_matrix_that_is_not_one_hot(monkeypatch, tmp_path):
    (train, valid), bed, params = _write_inputs(tmp_path)
    fwd = np.load(train)["fwd"]
    fwd[:, 20] = 0
    np.savez_compressed(train, fwd=fwd, hash=np.array(["0"]))
    monkeypatch.setattr(dgtrain, "training", lambda *a, **k: pytest.fail("must not train"))
    with pytest.raises(ValueError, match="one-hot"):
        cli.CommandLineParser().parse_args(["train", params, train, valid, bed]).run()


def test_chromosome_name():
    assert cli.chromosome_name("/data/chr1.fa.gz.npz") == "chr1"
    assert cli.chromosome_name("chrX_random.npz") == "chrX_random"


def test_train_without_its_arguments_is_a_usage_error():
    with pytest.raises(SystemExit, match="usage"):
        cli.CommandLineParser.train(argparse.Namespace(), dgmodel.Options())
