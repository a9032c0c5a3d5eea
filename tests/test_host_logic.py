"""Host-side logic of the cnn_cort mirror that needs no GPU: options, parameter packing,
NIfTI round trip, training-set bookkeeping vs the reference golden vectors, the C-ABI
library's symbol table."""
import configparser
import ctypes
import os
import pickle
import re

import numpy as np
import pytest

from cnn_cort import _native, nets, nifti, synthetic
from cnn_cort import base
from cnn_cort.load_options import device_index, load_options

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CFG = """
[database]
train_folder = /tmp/train
inference_folder = /tmp/test
t1_name = T1.nii.gz
roi_name = gt_15_classes.nii.gz
save_tmp = True

[model]
name = miccai2012_v1
mode = cuda0
patch_size = 32
batch_size = 256
patience = 20
net_verbose = 1
max_epochs = 100
train_split = 0.25
test_batch_size = 100000
load_weights = True
out_probabilities = False
speedup_segmentation = False
post_process = True
debug = True
"""


def _options():
    cfg = configparser.RawConfigParser()
    cfg.read_string(CFG)
    return load_options(cfg)


def test_load_options_keys_and_types():
    o = _options()
    assert o['experiment'] == 'miccai2012_v1' and o['patch_size'] == [32, 32]
    assert o['batch_size'] == 256 and o['test_batch_size'] == 100000 and o['train_split'] == 0.25
    assert o['load_weights'] == 'True' and o['debug'] == 'True' and o['post_process'] == 'True'
    assert o['crop'] == 'False' and o['crop_bool'] is False  # quirk Q2 fixed: parsed, not truthiness
    assert o['device'] == 0 and device_index('cuda3') == 3 and device_index('cpu') is None


def test_layer_table_matches_committed_pickle(weights_path):
    with open(weights_path, 'rb') as f:
        W = pickle.load(f, encoding='latin1')
    T = nets.layer_table()
    assert [n for n, _ in T] == list(W.keys())
    for n, shapes in T:
        assert [tuple(s) for s in shapes] == [a.shape for a in W[n]], n
    blob = nets.pack_params(W)
    assert blob.size == _native.PARAM_FLOATS == 883455
    P = nets.unpack_params(blob)
    for n in W:
        for a, b in zip(W[n], P[n]):
            assert np.array_equal(a, b)


def test_initial_params_follow_lasagne_defaults():
    P = nets._initial_params(seed=3)
    assert np.all(P['axial_ch_prelu1'][0] == 0.25) and np.all(P['FC1'][1] == 0)
    beta, gamma, mean, inv_std = P['coronal_ch_conv3_bn']
    assert not beta.any() and np.all(gamma == 1) and not mean.any() and np.all(inv_std == 1)
    lim = np.sqrt(6.0 / (20 * 9 + 40 * 9))
    w = P['axial_ch_conv3'][0]
    assert w.shape == (40, 20, 3, 3) and np.abs(w).max() <= lim and np.abs(w).max() > 0.9 * lim


def test_train_split_is_first_stratified_fold():
    y = np.array([0] * 8 + [1] * 5 + [2] * 4)
    tr, va = nets.TrainSplit(0.25).indices(y)
    assert list(va) == [0, 1, 8, 9, 13] and len(tr) + len(va) == len(y)
    assert set(tr).isdisjoint(va)


def test_generate_training_set_matches_reference(gather_golden):
    G = gather_golden
    n0 = 10
    args = ([G["B_x_axial"][:n0], G["B_x_axial"][n0:]], [G["B_x_coronal"][:n0], G["B_x_coronal"][n0:]],
            [G["B_x_saggital"][:n0], G["B_x_saggital"][n0:]], [G["T_atlas0"], G["T_atlas1"]],
            [G["B_y_axial"][:n0], G["B_y_axial"][n0:]])
    r = base.generate_training_set(*args, {"debug": "False"}, randomize=False)
    for k, v in zip(("xa", "xc", "xs", "at", "y"), r):
        assert v.dtype == G["T_plain_" + k].dtype and np.array_equal(v, G["T_plain_" + k]), k
    np.random.seed(77)
    r = base.generate_training_set(*args, {"debug": "False"}, randomize=True)
    for k, v in zip(("xa", "xc", "xs", "at", "y"), r):
        assert np.array_equal(v, G["T_shuf_" + k]), k


def test_nifti_round_trip(tmp_path):
    rng = np.random.RandomState(0)
    aff = np.array([[0.7, 0, 0, -10], [0, 0.7, 0, 5], [0, 0, 0.7, 2], [0, 0, 0, 1.0]])
    for arr in (rng.rand(5, 6, 7).astype(np.float32), rng.randint(0, 16, (4, 3, 2)).astype(np.uint8),
                rng.rand(3, 4, 5, 15).astype(np.float32), rng.randn(4, 4, 4)):
        for ext in (".nii", ".nii.gz"):
            p = str(tmp_path / ("a" + ext))
            nifti.Nifti1Image(arr, aff).to_filename(p)
            img = nifti.load(p)
            assert img.shape == arr.shape and img.get_data().dtype == arr.dtype
            assert np.array_equal(img.get_data(), arr) and np.allclose(img.affine, aff, atol=1e-6)


def test_synthetic_subject_and_test_names(tmp_path):
    d = synthetic.write_subject(str(tmp_path), "s01", shape=(40, 36, 32), seed=5, with_labels=True)
    t1 = nifti.load(os.path.join(d, "T1.nii.gz")).get_data()
    atlas = nifti.load(os.path.join(d, "tmp", "MNI_sub_probabilities.nii.gz")).get_data()
    lab = nifti.load(os.path.join(d, "gt_15_classes.nii.gz")).get_data()
    assert t1.shape == (40, 36, 32) and (t1 > 0).all() and atlas.shape == (40, 36, 32, 15)
    assert atlas.min() >= 0 and atlas.sum(-1).max() <= 1.0 + 1e-5
    assert lab.max() == 15 and ((lab > 0) & (lab < 15)).any()
    names, subj = base.load_test_names({"test_folder": str(tmp_path), "t1_name": "T1.nii.gz"})
    assert subj == ["s01"] and names[0].endswith("s01/T1.nii.gz")
    m = np.zeros((9, 9, 9), bool)
    m[2:4, 3:7, 5] = True
    assert base.bounding_box(m) == (2, 4, 3, 7, 5, 6) and base.bounding_box(np.zeros((2, 2, 2), bool)) is None


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads on a CPU-only box and exports everything include/*.h declares."""
    hdr = open(os.path.join(ROOT, "include", "subcort_b200.h")).read()
    declared = set(re.findall(r"SC_API [^;(]*?\b(sc_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 23
    assert declared == set(_native.PROTOTYPES), declared ^ set(_native.PROTOTYPES)
    if not os.path.exists(_native.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _native.load_library().sc_version() >= 100


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_native.NativeError, match="no CUDA device|CUDA"):
        _native.Context(0)
    with pytest.raises(_native.NativeError):
        nets.Net({'mode': 'cpu', 'patch_size': [32, 32]}, None, None)


def test_bench_reference_arm_prints_one_json_line():
    """bench.py contract: exactly one JSON line on stdout (library chatter goes to stderr); the reference arm runs the
    oracle port of the reference's mode=cpu path on the host cores, no GPU needed."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-sample", "128", "--size", "48"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "voxels/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
