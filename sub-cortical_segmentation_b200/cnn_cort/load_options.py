"""Options loader -- same keys and value types as the reference's
``cnn_cort/load_options.py:11-59`` (strings stay strings: 'True' / 'False').

Differences, all deliberate (SURVEY.md 5.6):
* ``mode = cudaN`` selects GPU N for the sm_100a kernels instead of setting THEANO_FLAGS;
  any other mode ('cpu') has no implementation here (the reference's CPU path exists only
  as the oracle/baseline) and build_model raises.
* ``options['crop']`` keeps the raw string for fidelity, and ``options['crop_bool']`` holds
  the parsed value: the reference tests the string's truthiness (base.py:367), so
  ``speedup_segmentation = False`` still cropped there (quirk Q2); here it does not.
"""
import configparser
import math


def _truthy(s):
    return str(s).strip().lower() in ("true", "1", "yes", "on")


def load_options(user_config):
    """map options from a ConfigParser into the flat options dict"""
    g = user_config.get
    options = {}
    options['experiment'] = g('model', 'name').strip()
    options['train_folder'] = g('database', 'train_folder').strip()
    options['test_folder'] = g('database', 'inference_folder').strip()
    options['output_folder'] = ''
    options['current_scan'] = ''
    options['t1_name'] = g('database', 't1_name').strip()
    options['roi_name'] = g('database', 'roi_name').strip()
    options['out_name'] = 'out_seg.nii.gz'
    options['save_tmp'] = g('database', 'save_tmp').strip()

    options['mode'] = g('model', 'mode').strip()
    ps = user_config.getint('model', 'patch_size')
    options['patch_size'] = [ps, ps]
    options['weight_paths'] = None
    options['train_split'] = user_config.getfloat('model', 'train_split')
    options['max_epochs'] = user_config.getint('model', 'max_epochs')
    options['patience'] = user_config.getint('model', 'patience')
    options['batch_size'] = user_config.getint('model', 'batch_size')
    options['test_batch_size'] = user_config.getint('model', 'test_batch_size')
    options['net_verbose'] = user_config.getint('model', 'net_verbose')
    options['load_weights'] = g('model', 'load_weights').strip()
    options['randomize_train'] = True
    options['debug'] = g('model', 'debug').strip()
    options['out_probabilities'] = g('model', 'out_probabilities').strip()
    options['post_process'] = g('model', 'post_process').strip()
    options['crop'] = g('model', 'speedup_segmentation').strip()
    options['crop_bool'] = _truthy(options['crop'])
    options['device'] = device_index(options['mode'])
    # optional: the template T1 and its [X,Y,Z,15] priors (on the template's grid) that register_masks maps onto subjects
    # whose tmp/ files are missing; without them such subjects are an error, as before
    for key in ('atlas_template', 'atlas_priors'):
        v = g('database', key, fallback='').strip()
        options[key] = v or None
    # optional: Monte-Carlo dropout passes of the dense inference (0 = off) and the seed of their masks
    for key in ('mc_samples', 'mc_seed'):
        v = user_config.getint('model', key, fallback=0)
        if v < 0:
            raise ValueError("[model] %s = %d must not be negative" % (key, v))
        options[key] = v
    # optional: fine-tune the head of a trained experiment's weights (nets/<fine_tune_from>/) on this experiment's training set
    # with the convolutional trunk frozen (Net.fine_tune) instead of training from scratch; off when absent or empty
    v = g('model', 'fine_tune_from', fallback='').strip()
    options['fine_tune_from'] = v or None
    if options['fine_tune_from'] == options['experiment']:
        raise ValueError("[model] fine_tune_from = %s names this experiment: its weights would be overwritten" % v)
    # optional: the isotropic voxel size (mm) the network runs on; the scan is resampled to it and the outputs mapped back to
    # the scan's grid (base.segment_arrays).  Off when absent or empty
    v = g('model', 'resample_mm', fallback='').strip()
    options['resample_mm'] = parse_resample_mm(v) if v else None
    # optional: training-time augmentation of the device-resident training set (Net.fit / Net.fine_tune on a ScanTrainingSet):
    # per sample a random rotation and scale about the centre voxel, contrast, brightness and Gaussian noise.  Off (None) when
    # every range is absent or 0
    options['augment'] = parse_augment({key: g('model', 'augment_' + key, fallback='').strip() for key in AUGMENT_KEYS})
    return options


# [model] augment_<key>: (lowest value, highest value, highest value allowed itself) of each range, the sc_augment contract
AUGMENT_RANGES = {'rotation_deg': (0.0, 180.0, True), 'scale': (0.0, math.inf, False), 'intensity': (0.0, 1.0, False),
                  'noise': (0.0, math.inf, False)}
AUGMENT_KEYS = tuple(AUGMENT_RANGES) + ('seed',)


def parse_augment(values):
    """{rotation_deg, scale, intensity, noise, seed: string or ''} -> the augmentation dict, or None when every range is 0
    or absent; a value that is not a number, not finite or out of its range raises ValueError"""
    aug = {}
    for key, (lo, hi, hi_ok) in AUGMENT_RANGES.items():
        v = values.get(key, '')
        try:
            x = float(v) if v != '' else 0.0
        except (TypeError, ValueError):
            raise ValueError("[model] augment_%s = %r is not a number" % (key, v))
        if not math.isfinite(x) or x < lo or x > hi or (x == hi and not hi_ok):
            raise ValueError("[model] augment_%s = %r must be finite and in [%g, %g%s" % (key, v, lo, hi, ']' if hi_ok else ')'))
        aug[key] = x
    v = values.get('seed', '')
    try:
        seed = int(v) if v != '' else 0
    except (TypeError, ValueError):
        raise ValueError("[model] augment_seed = %r is not an integer" % (v,))
    if not 0 <= seed < 1 << 64:
        raise ValueError("[model] augment_seed = %r must be in [0, 2^64)" % (v,))
    if not any(aug.values()):
        return None
    aug['seed'] = seed
    return aug


def parse_resample_mm(v):
    """a finite voxel size > 0 in mm, else ValueError"""
    try:
        mm = float(v)
    except (TypeError, ValueError):
        raise ValueError("[model] resample_mm = %r is not a number" % (v,))
    if not math.isfinite(mm) or mm <= 0:
        raise ValueError("[model] resample_mm = %r must be a finite number > 0" % (v,))
    return mm


def device_index(mode):
    """'cuda0' -> 0, 'cuda' -> 0; anything without 'cuda' -> None (no GPU requested)."""
    mode = str(mode).strip()
    if mode.find('cuda') == -1:
        return None
    digits = ''.join(ch for ch in mode if ch.isdigit())
    return int(digits) if digits else 0


def read_config(path):
    cfg = configparser.RawConfigParser()
    if not cfg.read(path):
        raise IOError("cannot read configuration file %s" % path)
    return load_options(cfg)


def print_options(options):
    print("--------------------------------------------------")
    print(" ")
    for k in options.keys():
        print(k, ':', options[k])
    print("--------------------------------------------------")
