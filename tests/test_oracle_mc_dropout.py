"""Monte-Carlo dropout oracle (sc_segment_volume_mc; tests/mc_dropout_oracle.py): the keep masks, the equivalence of masked
activations with row-masked weights that the device relies on, and the configuration keys."""
import configparser
import os
from collections import OrderedDict

import numpy as np
import pytest
import torch

from oracle import network
import mc_dropout_oracle as mco

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (seed, idx, hash3(seed, idx)) printed by the C++ function of csrc/common.cuh
HASH3_PINS = [(0, 0, 2822339357), (0, 1, 2657788345), (0, 2699, 3383786352), (7, 2700, 1797410863), (12345, 54321, 1573428299),
              (18446744073709551615, 1000000, 1467893583), (42, 1 << 40, 2383338452)]


def test_hash3_matches_the_cpp_function():
    for seed, idx, want in HASH3_PINS:
        assert int(mco.hash3(seed, idx)) == want, (seed, idx)
    idx = np.array([p[1] for p in HASH3_PINS[:3]], np.uint64)
    assert list(mco.hash3(0, idx)) == [p[2] for p in HASH3_PINS[:3]]


def test_keep_masks_layout_and_rate():
    k = mco.mc_keep_masks(3, 64)
    assert k.shape == (64, 2700) and k.dtype == np.uint8 and set(np.unique(k)) <= {0, 1}
    assert abs(k.mean() - 0.5) < 0.01
    assert k[5, 17] == mco.hash3(3, 5 * 2700 + 17) & 1              # pass t = the training step's sample t
    assert np.array_equal(mco.mc_keep_masks(3, 8), k[:8])           # passes do not depend on T
    assert not np.array_equal(mco.mc_keep_masks(4, 8), k[:8])


def _row_masked(P, keep):
    """P with the dense-layer weight rows of every dropout input scaled by 2 keep (pickle layout); fc_2's atlas rows as is."""
    s = 2.0 * keep.astype(np.float32)
    Q = OrderedDict((n, [a.copy() for a in arrs]) for n, arrs in P.items())
    for i, b in enumerate(mco.BRANCHES):
        Q["%s_d1" % b][0] *= s[i * 540:(i + 1) * 540, None]
    Q["FC1"][0] *= s[1620:2160, None]
    Q["fc_2"][0][:540] *= s[2160:2700, None]
    return Q


def test_dropout_pass_equals_row_masked_weights(oracle_params):
    rng = np.random.RandomState(4)
    n = 6
    x = [rng.randn(n, 1, 32, 32).astype(np.float32) for _ in range(3)]
    at = rng.dirichlet(np.ones(15) * 0.3, size=n).astype(np.float32)
    for seed, t in ((0, 0), (9, 5)):
        keep = mco.mc_keep_masks(seed, t + 1)[t]
        got = mco.forward_dropout(oracle_params, *x, at, keep)
        ref = network.forward(_row_masked(oracle_params, keep), *x, at, dtype=torch.float64)
        assert np.abs(got - ref).max() < 1e-12
    ones = np.ones(2700, np.uint8)        # keeping everything doubles every dropout input: not the deterministic net
    assert np.abs(mco.forward_dropout(oracle_params, *x, at, ones) -
                  network.forward(oracle_params, *x, at, dtype=torch.float64)).max() > 1e-3


def test_mc_predict_statistics(oracle_params):
    rng = np.random.RandomState(8)
    n = 5
    x = [rng.randn(n, 1, 32, 32).astype(np.float32) for _ in range(3)]
    at = rng.dirichlet(np.ones(15) * 0.3, size=n).astype(np.float32)
    pbar, H, mi = mco.mc_predict(oracle_params, *x, at, seed=2, T=3)
    keep = mco.mc_keep_masks(2, 3)
    passes = [mco.forward_dropout(oracle_params, *x, at, keep[t]) for t in range(3)]
    assert np.abs(pbar - np.mean(passes, 0)).max() < 1e-14
    assert np.abs(H + (pbar * np.log(pbar)).sum(1)).max() < 1e-12
    assert (mi >= 0).all() and (mi <= H).all() and (H <= np.log(15)).all()
    _, H1, mi1 = mco.mc_predict(oracle_params, *x, at, seed=2, T=1)
    assert (mi1 == 0).all() and (H1 > 0).all()


def _config(**model):
    cfg = configparser.RawConfigParser()
    assert cfg.read(os.path.join(ROOT, "configuration.cfg"))
    for k, v in model.items():
        cfg.set("model", k, str(v))
    return cfg


def test_load_options_mc_keys():
    from cnn_cort.load_options import load_options
    o = load_options(_config())
    assert o["mc_samples"] == 0 and o["mc_seed"] == 0               # old configuration files: off
    o = load_options(_config(mc_samples=8, mc_seed=11))
    assert o["mc_samples"] == 8 and o["mc_seed"] == 11
    for key in ("mc_samples", "mc_seed"):
        with pytest.raises(ValueError, match=key):
            load_options(_config(**{key: -1}))
