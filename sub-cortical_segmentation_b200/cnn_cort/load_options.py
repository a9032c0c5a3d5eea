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
    return options


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
