#!/usr/bin/env python
"""Example driver -- the Python 3 counterpart of the reference's train_model.py (same calls, same configuration.cfg
keys); everything below the imports runs on the B200 kernels.

    python train_model.py [configuration.cfg] [--train] [--evaluate]

--train with [model] fine_tune_from = <experiment> fine-tunes the head of nets/<experiment>/<experiment>.pkl on the training
folder (frozen convolutional trunk, Net.fine_tune) instead of training from scratch.
With [model] resample_mm set, training runs on the device-resident set resampled to that isotropic grid, as test_scan
segments.  With [model] augment_* ranges set, training runs on the device-resident set too, and every training minibatch is
gathered through random per-sample rotations, scales, contrast, brightness and noise.

--evaluate scores each inference subject that has manual labels (<subject>/<roi_name>): per-structure Dice and
surface distances of the segmentation test_scan wrote, and with [model] mc_samples > 0 the mean Monte-Carlo dropout entropy
inside each predicted structure.
"""
import configparser
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "sub-cortical_segmentation_b200"))

from cnn_cort.base import (evaluate_scan, generate_training_set, load_data, load_scan_training_set, load_test_names,  # noqa: E402
                           structure_uncertainty, test_scan)
from cnn_cort.nifti import load as load_nii  # noqa: E402
from cnn_cort.load_options import load_options, print_options  # noqa: E402
from cnn_cort.nets import build_model  # noqa: E402


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    cfg_path = args[0] if args else os.path.join(os.getcwd(), "configuration.cfg")
    user_config = configparser.RawConfigParser()
    if not user_config.read(cfg_path):
        raise SystemExit("cannot read %s" % cfg_path)
    options = load_options(user_config)
    print_options(options)
    weights_path = os.path.join(os.getcwd(), "nets")

    if "--train" in sys.argv and options['fine_tune_from']:
        # supervised domain adaptation: start from another experiment's weights, retrain the head on this training set with the
        # convolutional trunk frozen; the best weights land in nets/<name>/<name>.pkl as after fit
        net = build_model(weights_path, dict(options, load_weights='False'))
        src = os.path.join(weights_path, options['fine_tune_from'], options['fine_tune_from'] + '.pkl')
        print("    --> fine-tuning the head of", src)
        net.load_params_from(src)
        net.fine_tune(load_scan_training_set(options))
    elif "--train" in sys.argv and (options['resample_mm'] is not None or options['augment'] is not None):
        # on the network's grid: the device-resident set resamples every subject as test_scan does (load_data cannot); the
        # augmented gather cuts every minibatch from the scans (the patch arrays of load_data are already cut)
        net = build_model(weights_path, options)
        net.fit(load_scan_training_set(options))
    elif "--train" in sys.argv:
        x_axial, x_cor, x_sag, y, x_atlas, names = load_data(options)
        x_train_axial, x_train_cor, x_train_sag, x_train_atlas, y_train = generate_training_set(
            x_axial, x_cor, x_sag, x_atlas, y, options)
        net = build_model(weights_path, options)
        net.fit({'in1': x_train_axial, 'in2': x_train_cor, 'in3': x_train_sag, 'in4': x_train_atlas}, y_train)

    t1_test_paths, folder_names = load_test_names(options)
    options['net_verbose'] = 0
    net = build_model(weights_path, options)
    for t1, current_scan in zip(t1_test_paths, folder_names):
        t = test_scan(net, t1, options)
        print("    -->  tested subject :", current_scan, "(elapsed time:", t, "min.)")
        if "--evaluate" in sys.argv:
            print_evaluation(t1, options)


def print_evaluation(t1_path, options):
    """Score the segmentation test_scan wrote for one subject against its manual labels (<subject>/<roi_name>), if any."""
    subject_dir = os.path.dirname(t1_path)
    ref_path = os.path.join(subject_dir, options['roi_name'])
    if not os.path.exists(ref_path):
        return
    out_name = 'out_subcortical_seg_prec.nii.gz' if options['post_process'] == 'True' else 'out_subcortical_rawseg.nii.gz'
    seg_path = os.path.join(subject_dir, out_name)
    metrics, _ = evaluate_scan(seg_path, ref_path, device=options.get('device'))
    # Monte-Carlo dropout outputs of test_scan: the mean entropy inside each predicted structure, beside its Dice
    ent_path, mi_path = (os.path.join(subject_dir, f) for f in ('out_subcortical_entropy.nii.gz', 'out_subcortical_mi.nii.gz'))
    unc = None
    if os.path.exists(ent_path) and os.path.exists(mi_path):
        unc = structure_uncertainty(load_nii(seg_path).get_data(), load_nii(ent_path).get_data(), load_nii(mi_path).get_data(),
                                    device=options.get('device'))
    print("    -->  %s vs %s" % (out_name, options['roi_name']))
    print("         %9s %9s %9s %7s %9s %9s %9s%s" % ("structure", "n_seg", "n_ref", "dice", "hd_mm", "hd95_mm", "assd_mm",
                                                   " %9s" % "entropy" if unc else ""))
    for l, m in metrics.items():
        print("         %9d %9d %9d %7.4f %9.3f %9.3f %9.3f%s" % (l, m['n_seg'], m['n_ref'], m['dice'], m['hd_mm'], m['hd95_mm'],
                                                              m['assd_mm'], " %9.4f" % unc[l]['entropy'] if unc else ""))
    dice = [m['dice'] for m in metrics.values() if m['dice'] == m['dice']]
    print("         mean dice %.4f over %d structures" % (sum(dice) / len(dice) if dice else float('nan'), len(dice)))


if __name__ == "__main__":
    main()
