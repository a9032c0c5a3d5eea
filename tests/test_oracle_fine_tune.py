"""The fp64 reference of fine-tuning (tests/fine_tune_oracle.py) against the unchanged network oracle, by finite differences,
and the [model] fine_tune_from option."""
import configparser
import os

import numpy as np
import pytest
import torch

import fine_tune_oracle as fto
from oracle import network as on

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _batch(n, seed):
    rng = np.random.RandomState(seed)
    x = [rng.randn(n, 1, 32, 32).astype(np.float32) for _ in range(3)]
    at = rng.dirichlet(np.ones(15) * 0.3, size=n).astype(np.float32)
    y = rng.randint(0, 15, n).astype(np.uint8)
    masks = {"%s_l1drop" % b: (rng.rand(n, 60, 3, 3) < 0.5).astype(np.uint8) for b in on.BRANCHES}
    masks["f1_drop"] = (rng.rand(n, 540) < 0.5).astype(np.uint8)
    masks["f2_drop"] = (rng.rand(n, 540) < 0.5).astype(np.uint8)
    return x, at, y, masks


def test_head_on_trunk_features_is_the_network(oracle_params):
    x, at, _, _ = _batch(6, 1)
    feats = fto.trunk_features(oracle_params, *x)
    assert feats.shape == (6, 3, 540) and feats.dtype == np.float64
    ref = on.forward(oracle_params, *x, at, dtype=torch.float64)
    assert np.abs(fto.head_forward(oracle_params, feats, at) - ref).max() < 1e-12


def test_head_step_gradients_match_finite_differences():
    P = on.init_params(4)
    x, at, y, masks = _batch(5, 2)
    feats = fto.trunk_features(P, *x)
    loss, G, newP, state = fto.head_train_step(P, feats, at, y, masks=masks)
    assert abs(loss - fto.head_loss(P, feats, at, y, masks)) < 1e-12
    assert set(G) == set(fto.head_names(P)) and not any(fto.is_trunk(n) for n, _ in G)
    rng = np.random.RandomState(0)
    h = 1e-6
    for (name, k), g in G.items():
        flat = np.asarray(P[name][k], np.float64).reshape(-1)
        for j in rng.choice(flat.size, size=min(4, flat.size), replace=False):
            fd = []
            for s in (h, -h):
                Q = {n: [np.array(a, np.float64, copy=True) for a in arrs] for n, arrs in P.items()}
                Q[name][k].reshape(-1)[j] += s
                fd.append(fto.head_loss(Q, feats, at, y, masks))
            num = (fd[0] - fd[1]) / (2 * h)
            assert abs(num - g.reshape(-1)[j]) < 1e-6 + 1e-4 * abs(num), (name, k, j, num, g.reshape(-1)[j])
    assert state["t"] == 1


def test_head_step_copies_the_trunk():
    P = on.init_params(5)
    x, at, y, masks = _batch(4, 3)
    _, G, newP, _ = fto.head_train_step(P, fto.trunk_features(P, *x), at, y, masks=masks)
    moved = 0
    for name, arrs in P.items():
        for k, a in enumerate(arrs):
            if fto.is_trunk(name):
                assert np.array_equal(newP[name][k], a), name
            else:
                moved += not np.array_equal(newP[name][k], a)
    assert moved == len(G)


def _config(**model):
    cfg = configparser.RawConfigParser()
    assert cfg.read(os.path.join(ROOT, "configuration.cfg"))
    for k, v in model.items():
        cfg.set("model", k, str(v))
    return cfg


def test_load_options_fine_tune_from():
    from cnn_cort.load_options import load_options
    assert load_options(_config())["fine_tune_from"] is None                 # old configuration files: off
    assert load_options(_config(fine_tune_from=""))["fine_tune_from"] is None
    o = load_options(_config(name="site_b", fine_tune_from=" miccai2012_v1 "))
    assert o["fine_tune_from"] == "miccai2012_v1" and o["experiment"] == "site_b"
    name = load_options(_config())["experiment"]
    with pytest.raises(ValueError, match="fine_tune_from"):
        load_options(_config(fine_tune_from=name))
