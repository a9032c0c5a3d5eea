"""Data layer with the reference's signatures (``cnn_cort/base.py``), on the GPU.

Kept names: load_data, load_test_names, generate_training_set, load_patch_vectors,
get_atlas_vectors, load_patches, get_patches, get_mask_voxels, load_patch_batch, test_scan,
post_process_segmentation.  Candidate indexing, patch / atlas gathering, the network and the
result scatter and the 10x dilation of the crop mask run in ``libsubcort_b200.so``; NIfTI
I/O, intensity normalisation and the connected-component post-processing stay on the host
exactly where the reference has them (outside the timed path).

Deliberate deviations from reference quirks (SURVEY.md 5.6): Q1 prediction is not gated
by ``debug``; Q2 ``speedup_segmentation`` is parsed as a boolean; Q10 one forward pass
serves both labels and probabilities.  Registration (``register_masks``) runs on the device
(affine + B-spline NMI registration instead of niftyreg's binaries) when the configuration names a
template (``atlas_template`` / ``atlas_priors``); without one the ``tmp/MNI_*`` files must exist.
"""
import os
import random
import time

import numpy as np
from scipy import ndimage

from . import _native
from . import nifti as nib
from .nifti import load as load_nii

_contexts = {}


def get_context(device=None):
    """Process-wide sc_ctx per device for the data-layer helpers."""
    import torch
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if device not in _contexts:
        _contexts[device] = _native.Context(device)
    return _contexts[device]


def _dev(a, device, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a if dtype is None else a.astype(dtype, copy=False)))
    return t.to('cuda:%d' % device)


def _centers_tensor(centers, device):
    c = np.asarray(centers, dtype=np.int32).reshape(-1, 3)
    return _dev(c, device)


# ---------------------------------------------------------------------------------------------
# names
# ---------------------------------------------------------------------------------------------
def load_test_names(options):
    """Sorted sub-folders of the inference folder -> (T1 paths, subject names). [base.py:41-50]"""
    dir_name = options['test_folder']
    t1_name = options['t1_name']
    subjects = [f for f in sorted(os.listdir(dir_name)) if os.path.isdir(os.path.join(dir_name, f))]
    t1_names = [os.path.join(dir_name, subject, t1_name) for subject in subjects]
    return t1_names, subjects


# ---------------------------------------------------------------------------------------------
# candidates and patches
# ---------------------------------------------------------------------------------------------
def get_mask_voxels(mask, size=None, device=None, as_array=False):
    """Coordinates of the non-zero voxels in np.nonzero (C) order. [base.py:310-331]

    Returns a list of (x, y, z) tuples like the reference (``as_array=True``: int32 [N,3]).
    ``size``: shuffle (``random.shuffle``) and keep the first ``size`` entries.
    """
    ctx = get_context(device)
    m = np.asarray(mask)
    if m.dtype == np.bool_:
        m = m.view(np.uint8)
    elif m.dtype not in (np.uint8, np.float32, np.int32):
        m = (m != 0).view(np.uint8)
    xyz = ctx.nonzero_coords(_dev(m, ctx.device)).cpu().numpy()
    if size is not None:
        order = list(range(xyz.shape[0]))
        random.shuffle(order)
        xyz = xyz[order[:size]]
    if as_array:
        return xyz
    return [tuple(int(v) for v in r) for r in xyz]


def get_patches(image, centers, patch_size=(32, 32), mode='axial', device=None):
    """32x32 patches of one view around each centre, zeros outside the volume. [base.py:272-308]

    axial = [dx, dy] at z, coronal = [dx, dz] at y, saggital = [dy, dz] at x.
    Returns float32 [N, 32, 32] (the reference returns a list of N [32,32] arrays of the
    image dtype and every caller casts to float32; label volumes pass through exactly
    because labels <= 15 are exact in float32).
    """
    if tuple(patch_size) != (32, 32):
        raise ValueError("only patch_size (32, 32) is implemented")
    ctx = get_context(device)
    views = {'axial': (True, False, False), 'coronal': (False, True, False), 'saggital': (False, False, True)}[mode]
    vol = _dev(np.asarray(image), ctx.device, np.float32)
    out = ctx.gather_patches(vol, _centers_tensor(centers, ctx.device), views=views)
    return out[views.index(True)][:, 0].cpu().numpy()


def load_patch_batch(scan_name, options, datatype=np.float32):
    """Generator over test batches: (axial, coronal, saggital, atlas, centers). [base.py:335-397]

    Arrays are float32 [n,1,32,32] / [n,15] numpy like the reference's.  The volume and the
    atlas are uploaded once and stay on the device for the whole scan.
    """
    import torch
    ctx = get_context(options.get('device'))
    dir_name, name = os.path.split(scan_name)
    _ensure_registered(scan_name, options)
    image = load_nii(scan_name).get_data()
    atlas_name = os.path.join(dir_name, 'tmp', 'MNI_sub_probabilities.nii.gz')
    _require_registered(atlas_name)
    shape = tuple(int(s) for s in image.shape[:3])
    raw, dt = ctx.upload_volume(image)
    vol, _, _ = ctx.normalise_volume(raw, dt, shape)                       # base.py:358, numpy's result bit for bit
    if _crop_enabled(options):                                             # base.py:367-372
        mraw, mdt = ctx.upload_volume(nib.load(os.path.join(dir_name, 'tmp', 'MNI_subcortical_mask.nii.gz')).get_data())
        cand = ctx.dilate_mask(ctx.candidate_mask(mraw, mdt, shape), 10)
    else:
        cand = ctx.candidate_mask(raw, dt, shape)
    centers = ctx.nonzero_coords(cand)                                     # np.nonzero order, stays on the device
    if options['debug'] == 'True':
        print("    -->  num of samples to test:", len(centers))
    atlas = np.asarray(load_nii(atlas_name).get_data())
    if atlas.dtype != np.float32:
        atlas = atlas.astype(np.float32, order='K')
    d_atlas, _ = ctx.upload_volume(atlas, channels=15)
    d_atlas = d_atlas.view(torch.float32).view(shape + (15,))
    batch_size = options['test_batch_size']
    for i in range(0, len(centers), batch_size):
        c = centers[i:i + batch_size].contiguous()
        ax, co, sa, at = ctx.gather_patches(vol, c, atlas=d_atlas, bg_fix=True)
        yield (ax.cpu().numpy().astype(datatype, copy=False), co.cpu().numpy().astype(datatype, copy=False),
               sa.cpu().numpy().astype(datatype, copy=False), at.cpu().numpy(), [tuple(int(v) for v in r) for r in c.cpu().numpy()])


def normalise_test(image):
    """(image - mean_nz) / std_nz with numpy's own dtype promotion. [base.py:358]"""
    nz = image[np.nonzero(image)]
    return (image - nz.mean()) / nz.std()


def _crop_enabled(options):
    crop = options.get('crop_bool')
    if crop is None:
        crop = str(options.get('crop', 'True')).strip().lower() in ('true', '1', 'yes', 'on')
    return bool(crop)


def candidate_mask(image, dir_name, options):
    """bool volume of the voxels to classify. [base.py:367-372]"""
    if _crop_enabled(options):
        mask_atlas = nib.load(os.path.join(dir_name, 'tmp', 'MNI_subcortical_mask.nii.gz')).get_data()
        ctx = get_context(options.get('device'))
        m = _dev(np.ascontiguousarray(mask_atlas != 0).view(np.uint8), ctx.device)
        return ctx.dilate_mask(m, 10).cpu().numpy().astype(bool)   # == ndimage.binary_dilation(mask, iterations=10)
    return image.astype(bool)


def _require_registered(atlas_name):
    if not os.path.exists(atlas_name):
        raise IOError("%s is missing: atlas registration (register_masks / niftyreg) is outside this "
                      "implementation's scope -- create the tmp/MNI_* files with the reference pipeline" % atlas_name)


_REGISTERED = ('MNI_sub_probabilities.nii.gz', 'MNI_subcortical_mask.nii.gz')


def _ensure_registered(t1_path, options):
    """register_masks for a subject whose tmp/MNI_* files are missing, when the configuration names a template; -> the
    device-resident (priors, mask) it produced, or None (files present, or no template: the callers then raise)"""
    tmp = os.path.join(os.path.dirname(t1_path), 'tmp')
    if all(os.path.exists(os.path.join(tmp, n)) for n in _REGISTERED):
        return None
    if not (options.get('atlas_template') and options.get('atlas_priors')):
        return None
    return register_masks(t1_path, options)


# ---------------------------------------------------------------------------------------------
# inference
# ---------------------------------------------------------------------------------------------
def test_scan(net, test_scan, options):
    """Segment one scan and write the reference's output files; returns elapsed minutes.
    [base.py:401-458]

    options['inference'] = 'dense' (default): whole-volume dilated formulation restricted to
    the bounding box of the candidates (sc_segment_volume); 'patchwise': the reference's own
    flow, batch by batch through net.predict / predict_proba on gathered patches.
    """
    s_time = time.time()
    image_path, name = os.path.split(test_scan)
    mode = options.get('inference', 'dense')
    # I/O: in the dense mode the files are read straight into page-locked memory, in the array order they have on disk
    t1_nii = nib.load(test_scan, pinned=(mode != 'patchwise'))
    t1 = t1_nii.get_data()
    want_proba = options['out_probabilities'] == 'True'
    mc_samples = int(options.get('mc_samples', 0) or 0)
    mc = {'samples': mc_samples, 'seed': int(options.get('mc_seed', 0) or 0)} if mc_samples > 0 else None
    if mode == 'patchwise':
        if mc is not None:
            raise ValueError("mc_samples = %d: Monte-Carlo dropout is implemented for the dense inference mode only" % mc_samples)
        image = np.zeros_like(t1)
        image_proba = np.zeros(t1_nii.shape + (15,)) if want_proba else None
        for batch_axial, batch_cor, batch_sag, atlas, centers in load_patch_batch(test_scan, options):
            X = {'in1': batch_axial, 'in2': batch_cor, 'in3': batch_sag, 'in4': atlas}
            x, y, z = np.stack(centers, axis=1)
            if want_proba:
                y_pred_proba = net.predict_proba(X)
                image[x, y, z] = np.argmax(y_pred_proba, axis=1)
                image_proba[x, y, z, :] = y_pred_proba
            else:
                image[x, y, z] = net.predict(X)
    else:
        timings = options.get('timings')
        registered = _ensure_registered(test_scan, options)
        if registered is not None:                 # the priors and mask just registered stay on the device
            atlas, mask = registered
            crop_mask = mask if _crop_enabled(options) else None
            post_mask = mask if options['post_process'] == 'True' else None
        else:
            atlas_name = os.path.join(image_path, 'tmp', 'MNI_sub_probabilities.nii.gz')
            _require_registered(atlas_name)
            atlas = nib.load(atlas_name, pinned=True).get_data()
            crop_mask = None
            if _crop_enabled(options):
                crop_mask = nib.load(os.path.join(image_path, 'tmp', 'MNI_subcortical_mask.nii.gz'), pinned=True).get_data()
            post_mask = None
            if options['post_process'] == 'True':      # filtered on the device, before the label volume is downloaded
                post_mask = crop_mask if crop_mask is not None else nib.load(os.path.join(image_path, 'tmp', 'MNI_subcortical_mask.nii.gz'), pinned=True).get_data()
        labels, image_proba, n_cand = segment_arrays(net.ctx, t1, atlas, crop_mask, want_proba, timings, post_mask=post_mask, mc=mc)
        if options['debug'] == 'True':
            print("    -->  num of samples to test:", n_cand)
        image = labels.astype(t1.dtype)

    if want_proba:
        nib.Nifti1Image(image_proba, affine=t1_nii.affine).to_filename(os.path.join(image_path, 'out_subcortical_prob.nii.gz'))
    if mc is not None:
        for key, fname in (('entropy', 'out_subcortical_entropy.nii.gz'), ('mutual_info', 'out_subcortical_mi.nii.gz')):
            nib.Nifti1Image(mc[key], affine=t1_nii.affine).to_filename(os.path.join(image_path, fname))
    if options['post_process'] == 'True':
        filtered = image if mode != 'patchwise' else post_process_segmentation(image_path, image, device=options.get('device'))
        nib.Nifti1Image(filtered, affine=t1_nii.affine).to_filename(os.path.join(image_path, 'out_subcortical_seg_prec.nii.gz'))
    else:
        nib.Nifti1Image(image, affine=t1_nii.affine).to_filename(os.path.join(image_path, 'out_subcortical_rawseg.nii.gz'))
    return (time.time() - s_time) / 60.0


def segment_arrays(ctx, t1, atlas, crop_mask=None, want_proba=False, timings=None, post_mask=None, mc=None):
    """The timed part of test_scan for one scan, device-resident from the first byte [base.py:357-372, 401-440]:
    raw T1 / atlas priors (/ registered mask) as host arrays in -> uint8 label volume (+ float32 [X,Y,Z,15] probabilities,
    number of candidates) out.  One upload per array (Fortran-ordered NIfTI arrays are reordered on the device), then
    normalisation over the non-zero voxels (numpy's result bit for bit), candidate mask (non-zero T1 voxels, or the
    registered mask dilated 10 times), its bounding box, the dense network pass and the scatter, all without the mask,
    the normalised volume or the coordinates ever visiting the host; one download of the result.  atlas / crop_mask /
    post_mask may also be CUDA tensors (float32 [X,Y,Z,15] C-ordered priors, [X,Y,Z] masks: what register_masks returns):
    they are used in place.

    mc={'samples': T, 'seed': s}: Monte-Carlo dropout (sc_segment_volume_mc) -- the labels and probabilities are those of the
    mean of T dropout passes, and on return the dict also holds 'entropy' (predictive entropy, nats) and 'mutual_info' as
    float32 [X,Y,Z] host arrays, zero outside the candidates."""
    import torch
    t0 = time.time()
    shape = tuple(int(s) for s in t1.shape[:3])
    on_device = torch.is_tensor(atlas)
    if not on_device:
        atlas = np.asarray(atlas)
        if atlas.dtype != np.float32:      # a scaled NIfTI comes back as float64: the priors are consumed as float32 (base.py:388)
            atlas = atlas.astype(np.float32, order='K')
    main = torch.cuda.current_stream()
    side = _side_stream(ctx.device)
    atlas_ready = torch.cuda.Event()
    d_atlas = None

    def device_bytes(a):
        """(C-ordered raw bytes on the device, dtype) of a host volume or a CUDA tensor"""
        if torch.is_tensor(a):
            return a.contiguous().view(-1).view(torch.uint8), np.dtype(str(a.dtype).replace('torch.', ''))
        return ctx.upload_volume(a)

    def start_atlas_upload(box):
        if on_device:
            return atlas
        # The priors (94 % of the upload) are first needed by the FC head: they are uploaded and reordered on a side stream while
        # the convolution phase runs -- enqueued behind the host-synchronous steps that precede it, whose small device -> host
        # copies would otherwise queue up behind the gigabyte.  Crop mode reads the priors at the candidates only: just the
        # bounding box of the dilated mask is uploaded (strided DMA from the host array).
        side.wait_stream(main)
        with torch.cuda.stream(side):
            if box is not None:
                d = ctx.upload_volume_box(atlas, box, channels=15)
            else:
                d, _ = ctx.upload_volume(atlas, channels=15)
                d = d.view(torch.float32).view(shape + (15,))
            atlas_ready.record(side)
        return d

    # T1 first: copies of one direction are served in issue order, and the convolution phase only waits for the T1 volume
    raw, dt = ctx.upload_volume(t1)
    vol, mean, std = ctx.normalise_volume(raw, dt, shape)
    if crop_mask is not None:
        mraw, mdt = device_bytes(crop_mask)
        cand = ctx.dilate_mask(ctx.candidate_mask(mraw, mdt, shape), 10)   # == ndimage.binary_dilation(mask, iterations=10)
    else:
        cand = ctx.candidate_mask(raw, dt, shape)                          # == image.astype('bool')
    box, n_cand = ctx.mask_bbox(cand)
    if box is not None:
        d_atlas = start_atlas_upload(box if crop_mask is not None else None)
    lab = torch.zeros(shape, dtype=torch.uint8, device=vol.device)
    prob = torch.zeros(shape + (15,), dtype=torch.float32, device=vol.device) if want_proba else None
    ent = mi = None
    if mc is not None:
        ent = torch.zeros(shape, dtype=torch.float32, device=vol.device)
        mi = torch.zeros(shape, dtype=torch.float32, device=vol.device)
    if box is not None:
        ready = None if on_device else atlas_ready
        if mc is None:
            ctx.segment_volume(vol, d_atlas, box=box, cand_mask=cand, label_vol=lab, proba_vol=prob, atlas_ready=ready)
        else:
            ctx.segment_volume_mc(vol, d_atlas, int(mc['samples']), int(mc.get('seed', 0)), box=box, cand_mask=cand, label_vol=lab,
                                  proba_vol=prob, entropy_vol=ent, mi_vol=mi, atlas_ready=ready)
    main.wait_stream(side)
    if post_mask is not None:        # post_process_segmentation (base.py:460-480) on the device-resident label volume
        if post_mask is crop_mask and crop_mask is not None:
            pm = ctx.candidate_mask(mraw, mdt, shape)
        else:
            praw, pdt = device_bytes(post_mask)
            pm = ctx.candidate_mask(praw, pdt, shape)
        lab = ctx.post_process(lab, pm)
    h_lab = _pinned_out('lab', shape, torch.uint8)
    h_lab.copy_(lab, non_blocking=True)
    h_prob = None
    if want_proba:
        h_prob = _pinned_out('prob', shape + (15,), torch.float32)
        h_prob.copy_(prob, non_blocking=True)
    if mc is not None:
        mc['entropy'], mc['mutual_info'] = ent.cpu().numpy(), mi.cpu().numpy()
    torch.cuda.current_stream().synchronize()
    if timings is not None:
        timings.update({'hot_s': time.time() - t0, 'n_candidates': n_cand, 'mean_nz': mean, 'std_nz': std, 'box': box})
    # views of reusable page-locked buffers: valid until the next call
    return h_lab.numpy(), (h_prob.numpy() if want_proba else None), n_cand


def structure_uncertainty(labels, entropy, mutual_info, device=None):
    """Per-structure quality-control numbers of a Monte-Carlo dropout segmentation, on the device: for every label
    l = 1..14 the voxel count of the predicted structure and the mean predictive entropy and mean mutual information
    over its voxels (NaN for an empty structure).  labels [X,Y,Z] integral; entropy / mutual_info float [X,Y,Z]; host
    arrays or torch tensors.  -> {l: {'voxels': int, 'entropy': float, 'mutual_info': float}}"""
    import torch
    ctx = get_context(device)
    if not (tuple(labels.shape) == tuple(entropy.shape) == tuple(mutual_info.shape)) or len(labels.shape) != 3:
        raise ValueError("labels, entropy and mutual_info must be 3-D volumes of one shape, got %s, %s and %s" % (
            tuple(labels.shape), tuple(entropy.shape), tuple(mutual_info.shape)))
    d = 'cuda:%d' % ctx.device
    lab = _label_volume(labels, 'labels', ctx.device).view(-1).long()
    stats = []
    for v in (entropy, mutual_info):
        t = v if torch.is_tensor(v) else torch.from_numpy(np.ascontiguousarray(v))
        stats.append(torch.zeros(17, dtype=torch.float64, device=d).index_add_(0, lab, t.to(d, torch.float64).reshape(-1)))
    count = torch.bincount(lab, minlength=17).cpu().numpy()
    h, m = stats[0].cpu().numpy(), stats[1].cpu().numpy()
    nan = float('nan')
    return {l: {'voxels': int(count[l]), 'entropy': float(h[l] / count[l]) if count[l] else nan,
                'mutual_info': float(m[l] / count[l]) if count[l] else nan} for l in range(1, 15)}


_pinned_cache = {}
_side_streams = {}


def _side_stream(device):
    import torch
    if device not in _side_streams:
        _side_streams[device] = torch.cuda.Stream(device=device)
    return _side_streams[device]


def _pinned_out(key, shape, dtype):
    """reusable page-locked result buffers (allocating 1 GB of pinned memory per scan would cost more than the scan)"""
    import torch
    t = _pinned_cache.get(key)
    n = int(np.prod(shape))
    if t is None or t.dtype != dtype or t.numel() < n:
        t = torch.empty(n, dtype=dtype, pin_memory=True)
        _pinned_cache[key] = t
    return t[:n].view(shape)


def bounding_box(mask):
    """half-open (x0, x1, y0, y1, z0, z1) of the True voxels, or None"""
    if not mask.any():
        return None
    box = []
    for ax in range(3):
        other = tuple(a for a in range(3) if a != ax)
        nz = np.nonzero(mask.any(axis=other))[0]
        box += [int(nz[0]), int(nz[-1]) + 1]
    return tuple(box)


def post_process_segmentation(image_folder, input_mask, device=None):
    """Per label 1..14 keep the 6-connected component overlapping the registered sub-cortical mask most. [base.py:460-480]
    Runs on the device (sc_post_process: one union-find labelling pass for all classes), with the reference's quirks: a
    class without any component inside the mask selects "component 0", i.e. everything that is not of that class."""
    import torch
    ctx = get_context(device)
    atlas = load_nii(os.path.join(image_folder, 'tmp', 'MNI_subcortical_mask.nii.gz')).get_data()
    shape = tuple(int(s) for s in input_mask.shape[:3])
    seg = torch.from_numpy(np.ascontiguousarray(input_mask).astype(np.uint8)).to('cuda:%d' % ctx.device)
    mraw, mdt = ctx.upload_volume(atlas)
    mask = ctx.candidate_mask(mraw, mdt, shape)
    out = ctx.post_process(seg, mask)
    return out.cpu().numpy().astype(input_mask.dtype)


# ---------------------------------------------------------------------------------------------
# evaluation against manual labels
# ---------------------------------------------------------------------------------------------
def _label_volume(a, name, device):
    """label volume of any integer / float / bool dtype holding integral labels (numpy array or torch tensor) -> uint8
    CUDA tensor.  Labels above 15 become 16, so that sc_evaluate_segmentation rejects them and names the input."""
    import torch
    if torch.is_tensor(a):
        if a.dtype == torch.bool:
            a = a.to(torch.uint8)
        elif a.dtype != torch.uint8:
            if a.is_floating_point() and not bool((a == torch.floor(a)).all()):
                raise ValueError("%s holds non-integral labels" % name)
            if bool((a < 0).any()):
                raise ValueError("%s holds negative labels" % name)
            a = a.clamp(max=16).to(torch.uint8)
        return a.to('cuda:%d' % device).contiguous()
    a = np.asarray(a)
    if a.dtype != np.uint8:
        if a.dtype.kind == 'f' and not np.array_equal(a, np.floor(a)):
            raise ValueError("%s holds non-integral labels" % name)
        if a.dtype.kind not in 'fiub':
            raise TypeError("%s: unsupported label dtype %s" % (name, a.dtype))
        if a.dtype.kind in 'fi' and a.size and a.min() < 0:
            raise ValueError("%s holds negative labels" % name)
        a = np.minimum(a, 16).astype(np.uint8)
    return _dev(a, device)


def evaluate_segmentation(seg, ref, spacing=(1.0, 1.0, 1.0), device=None):
    """Score a segmentation against manual labels, on the device (sc_evaluate_segmentation).

    seg, ref: [X, Y, Z] label volumes with values 0..15 (15 counts as background), as host arrays of any integer or float
    dtype holding integral labels or as torch tensors; spacing: voxel size in mm along x, y, z.  Returns
    ({l: {field: value}} for the structures l = 1..14, confusion int64 [15, 15] indexed [ref class][seg class]).  Fields:
    n_seg, n_ref, n_both (voxel counts), dice (NaN when both are empty), vol_seg_mm3, vol_ref_mm3 and the surface distances
    hd_mm, hd95_mm, assd_mm (NaN when either structure is empty); definitions in include/subcort_b200.h."""
    ctx = get_context(device)
    if tuple(seg.shape) != tuple(ref.shape) or len(seg.shape) != 3:
        raise ValueError("seg and ref must be 3-D volumes of one shape, got %s and %s" % (tuple(seg.shape), tuple(ref.shape)))
    d_seg = _label_volume(seg, 'seg', ctx.device)
    d_ref = d_seg if ref is seg else _label_volume(ref, 'ref', ctx.device)
    rows, confusion = ctx.evaluate_segmentation(d_seg, d_ref, spacing, confusion=True)
    metrics = {l: {f: (int(rows[l - 1][f]) if f.startswith('n_') else float(rows[l - 1][f])) for f in rows.dtype.names}
               for l in range(1, 15)}
    return metrics, confusion


def evaluate_scan(seg_path, ref_path, device=None):
    """evaluate_segmentation of two NIfTI label files of one shape; the spacing is the reference's voxel size (the column
    norms of its affine, as nifti.py writes them)."""
    seg_nii, ref_nii = load_nii(seg_path), load_nii(ref_path)
    if tuple(seg_nii.shape) != tuple(ref_nii.shape):
        raise ValueError("%s and %s differ in shape: %s vs %s" % (seg_path, ref_path, seg_nii.shape, ref_nii.shape))
    spacing = tuple(float(s) for s in np.sqrt((np.asarray(ref_nii.affine)[:3, :3] ** 2).sum(0)))
    return evaluate_segmentation(seg_nii.get_data(), ref_nii.get_data(), spacing, device=device)


# ---------------------------------------------------------------------------------------------
# atlas registration
# ---------------------------------------------------------------------------------------------
def _cuda_f32(a, device):
    import torch
    if torch.is_tensor(a):
        return a.to('cuda:%d' % device, torch.float32).contiguous()
    return _dev(np.ascontiguousarray(a, dtype=np.float32), device)


def register_arrays(ctx, t1, t1_affine, template, template_affine, priors):
    """Map a template and its priors onto a subject on the device: affine then B-spline FFD registration of the template
    T1 to the subject T1 (NMI; sc_register_affine / sc_register_ffd), the priors warped through the result
    (sc_warp_volume) and the sub-cortical mask (sc_prior_mask: channels 0..12 summing to > 0, dilated 5 times).
    t1 / template: [X,Y,Z] volumes (host arrays or tensors; zeros in t1 are outside the subject), priors [X,Y,Z,15] on the
    template's grid, *_affine: 4x4 voxel -> mm.  -> CUDA tensors (affine float64 [4,4] subject mm -> template mm, grid
    float32 [gx,gy,gz,3], priors float32 [X,Y,Z,15] on the subject's grid, mask float32 0/1 [X,Y,Z])."""
    import torch
    ref, flo = _cuda_f32(t1, ctx.device), _cuda_f32(template, ctx.device)
    A = ctx.register_affine(ref, t1_affine, flo, template_affine)
    grid = ctx.register_ffd(ref, t1_affine, flo, template_affine, A)
    warped = ctx.warp_volume(_cuda_f32(priors, ctx.device), template_affine, A, grid, ref.shape, t1_affine)
    mask = ctx.prior_mask(warped, 5)
    return torch.from_numpy(A).to(ref.device), grid, warped, mask


def register_masks(t1_path, options, timings=None):
    """Register the configured template (options['atlas_template'], options['atlas_priors']) to the subject
    <subject>/<t1> and write what the reference's niftyreg calls leave in <subject>/tmp/ (base.py:483-551), with the
    subject's affine: transf.txt (4x4, subject mm -> template mm, the direction reg_aladin -aff writes),
    rT1d_template.nii.gz (the warped template T1), MNI_sub_probabilities.nii.gz ([X,Y,Z,15] priors) and
    MNI_subcortical_mask.nii.gz (float32 0/1).  Files that already exist are kept.  -> the device-resident
    (priors, mask) CUDA tensors.  timings (dict, optional) receives register_s and write_s."""
    template_path, priors_path = options.get('atlas_template'), options.get('atlas_priors')
    if not (template_path and priors_path):
        raise IOError("register_masks needs atlas_template and atlas_priors in the [database] section of the configuration")
    t0 = time.time()
    tmp = os.path.join(os.path.dirname(t1_path), 'tmp')
    os.makedirs(tmp, exist_ok=True)
    ctx = get_context(options.get('device'))
    t1_nii, tpl_nii, pri_nii = load_nii(t1_path), load_nii(template_path), load_nii(priors_path)
    if tuple(pri_nii.shape) != tuple(tpl_nii.shape[:3]) + (15,):
        raise ValueError("%s: priors of shape %s do not match the template %s (expected [X,Y,Z,15])" % (
            priors_path, tuple(pri_nii.shape), tuple(tpl_nii.shape)))
    A, grid, priors, mask = register_arrays(ctx, t1_nii.get_data(), t1_nii.affine, tpl_nii.get_data(), tpl_nii.affine,
                                            pri_nii.get_data())
    import torch
    torch.cuda.current_stream().synchronize()
    t1_s = time.time()
    aff = t1_nii.affine
    out = {'transf.txt': None, 'rT1d_template.nii.gz': None, 'MNI_sub_probabilities.nii.gz': priors, 'MNI_subcortical_mask.nii.gz': mask}
    for name, data in out.items():
        path = os.path.join(tmp, name)
        if os.path.exists(path):
            continue
        if name == 'transf.txt':
            np.savetxt(path, A.cpu().numpy())
        elif name == 'rT1d_template.nii.gz':
            warped = ctx.warp_volume(_cuda_f32(tpl_nii.get_data(), ctx.device), tpl_nii.affine, A.cpu().numpy(), grid, priors.shape, aff)
            nib.Nifti1Image(warped.cpu().numpy(), affine=aff).to_filename(path)
        else:
            nib.Nifti1Image(data.cpu().numpy(), affine=aff).to_filename(path)
    if timings is not None:
        timings.update({'register_s': t1_s - t0, 'write_s': time.time() - t1_s})
    return priors, mask


# ---------------------------------------------------------------------------------------------
# training data
# ---------------------------------------------------------------------------------------------
def load_data(options):
    """-> (x_axial, x_cor, x_sag, y_axial, x_atlas, names), lists indexed by subject.
    [base.py:11-37]"""
    _register_folder(options['train_folder'], options)
    (x_axial, y_axial, x_cor, y_cor, x_sag, y_sag, x_atlas, names) = load_patches(
        dir_name=options['train_folder'], t1_name=options['t1_name'], mask_name=options['roi_name'],
        size=tuple(options['patch_size']), device=options.get('device'))
    return x_axial, x_cor, x_sag, y_axial, x_atlas, names


def _register_folder(dir_name, options):
    for subject in sorted(os.listdir(dir_name)):
        if os.path.isdir(os.path.join(dir_name, subject)):
            _ensure_registered(os.path.join(dir_name, subject, options['t1_name']), options)


def load_patches(dir_name, mask_name, t1_name, size, seeds=None, balance_neg=True, device=None):
    """[base.py:221-256]"""
    print('    --> Loading ' + t1_name + ' images')
    x_axial, y_axial, x_cor, y_cor, x_sag, y_sag, centers, t1_names = load_patch_vectors(
        t1_name, mask_name, dir_name, size, balance_neg=balance_neg, device=device)
    x_atlas = get_atlas_vectors(dir_name, centers, t1_names, device=device)
    return x_axial, y_axial, x_cor, y_cor, x_sag, y_sag, x_atlas, t1_names


def _train_normalise(im):
    """float32 (im - mean_nz) / std_nz of the training path. [base.py:146]"""
    nz = im[np.nonzero(im)]
    # base.py:146 under the reference's numpy 1.12: a float32 array combined with float64 *scalars* stays float32
    # (value-based casting), i.e. the mean and std are rounded to float32 first; NumPy 2 would promote to float64
    return (im.astype(np.float32) - np.float32(nz.mean())) / np.float32(nz.std())


def _training_centres(mask, device, balance_neg=True):
    """int32 [n, 3]: every voxel with label 1..14 in np.nonzero order, then as many shuffled label-15 voxels (Python's
    ``random``, consumed as get_mask_voxels(..., size=len(pos)) does). [base.py:153-181]"""
    pos = get_mask_voxels(np.logical_and(mask > 0, mask < 15), device=device, as_array=True)
    neg = get_mask_voxels(mask == 15, size=len(pos) if balance_neg else None, device=device, as_array=True)
    return np.concatenate([pos, neg]).astype(np.int32)


def _training_order(n, randomize):
    """Row order of generate_training_set: None (concatenation order) or the permutation drawn from np.random. [base.py:98-110]"""
    if not randomize:
        return None
    seed = np.random.randint(np.iinfo(np.int32).max)
    # np.random.seed(seed); np.random.permutation(a) == a[RandomState(seed).permutation(len(a))]
    return np.random.RandomState(seed).permutation(n)


def load_patch_vectors(name, label_name, dir_name, size, random_state=42, balance_neg=True, device=None):
    """Boundary-restricted sampling per subject: every voxel with label 1..14 plus as many
    shuffled label-15 voxels; T1 patches of the three views and the label patches.
    [base.py:120-184]

    The reference gathers label patches for all three views only to read their centre pixel
    later (base.py:85); the returned y_* arrays are therefore [n, 32, 32] uint8 patches whose
    centre pixel holds the label gathered on the GPU and zeros elsewhere.
    """
    if tuple(size) != (32, 32):
        raise ValueError("only patch_size (32, 32) is implemented")
    ctx = get_context(device)
    subjects = [f for f in sorted(os.listdir(dir_name)) if os.path.isdir(os.path.join(dir_name, f))]
    image_names = [os.path.join(dir_name, subject, name) for subject in subjects]
    label_names = [os.path.join(dir_name, subject, label_name) for subject in subjects]
    x_axial, y_axial, x_cor, y_cor, x_sag, y_sag, vox_positions = [], [], [], [], [], [], []
    for image_name, lab_name in zip(image_names, label_names):
        im_norm = _train_normalise(load_nii(image_name).get_data())
        mask = load_nii(lab_name).get_data()
        cen = _training_centres(mask, ctx.device, balance_neg)
        vol = _dev(im_norm, ctx.device, np.float32)
        cdev = _centers_tensor(cen, ctx.device)
        ax, co, sa, _ = ctx.gather_patches(vol, cdev)
        lab = ctx.gather_center_labels(_dev(mask, ctx.device, np.uint8), cdev).cpu().numpy()
        ypatch = np.zeros((len(cen), 32, 32), np.uint8)
        ypatch[:, 16, 16] = lab
        x_axial.append(ax[:, 0].cpu().numpy()); x_cor.append(co[:, 0].cpu().numpy()); x_sag.append(sa[:, 0].cpu().numpy())
        y_axial.append(ypatch); y_cor.append(ypatch); y_sag.append(ypatch)
        vox_positions.append(cen)
    return x_axial, y_axial, x_cor, y_cor, x_sag, y_sag, vox_positions, image_names


def get_atlas_vectors(dir_name, centers, t1_names, device=None):
    """Atlas prior vector at every training centre, no background fix (the reference's fix
    there never fires, quirk Q4). [base.py:187-218]"""
    ctx = get_context(device)
    subjects = [f for f in sorted(os.listdir(dir_name)) if os.path.isdir(os.path.join(dir_name, f))]
    atlas_names = [os.path.join(dir_name, subject, 'tmp', 'MNI_sub_probabilities.nii.gz') for subject in subjects]
    out = []
    for atlas_name, c in zip(atlas_names, centers):
        _require_registered(atlas_name)
        atlas = load_nii(atlas_name).get_data()
        a = _dev(atlas, ctx.device, np.float32)
        dummy = a[..., 0].contiguous()
        res = ctx.gather_patches(dummy, _centers_tensor(c, ctx.device), atlas=a, bg_fix=False, views=(False, False, False))
        out.append(res[3].cpu().numpy().astype(atlas.dtype, copy=False))
    return out


def generate_training_set(x_axial, x_coronal, x_saggital, x_atlas, y, options, randomize=True):
    """Concatenate subjects, take the centre label, map 15 -> 0, shuffle everything with one
    seed, add the channel axis. [base.py:53-117]  Host-side: it is index bookkeeping."""
    x_train_axial = np.concatenate(x_axial, axis=0).astype('float32')
    x_train_cor = np.concatenate(x_coronal, axis=0).astype('float32')
    x_train_sag = np.concatenate(x_saggital, axis=0).astype('float32')
    x_train_atlas = np.concatenate(x_atlas, axis=0).astype('float32')
    y_train = np.concatenate(y, axis=0).astype('uint8')
    y_train = np.squeeze(y_train[:, y_train.shape[1] // 2, y_train.shape[2] // 2])
    y_train[y_train == 15] = 0
    perm = _training_order(len(y_train), randomize)
    if perm is not None:
        x_train_axial, x_train_cor, x_train_sag = x_train_axial[perm], x_train_cor[perm], x_train_sag[perm]
        y_train, x_train_atlas = y_train[perm], x_train_atlas[perm]
    x_train_axial = np.expand_dims(x_train_axial, axis=1)
    x_train_cor = np.expand_dims(x_train_cor, axis=1)
    x_train_sag = np.expand_dims(x_train_sag, axis=1)
    if options['debug'] == 'True':
        print("    --> X_TRAIN: ", x_train_axial.shape[0], x_train_axial.shape)
        print("    --> Y_TRAIN POS: ", y_train[y_train > 0].shape[0])
        print("    --> Y_TRAIN NEG: ", y_train[y_train == 0].shape[0])
    return x_train_axial, x_train_cor, x_train_sag, x_train_atlas, y_train


# ---------------------------------------------------------------------------------------------
# training data kept on the device: scans + sample table instead of patch arrays
# ---------------------------------------------------------------------------------------------
def check_sample_table(shapes, samples, atlas_rows, labels):
    """Reject a malformed training table before anything reaches the device: sc_gather_samples trusts its table.
    shapes: (X, Y, Z) per scan; samples: int [N, 4] (scan, x, y, z); atlas_rows: [N, 15]; labels: [N]."""
    samples, atlas_rows, labels = np.asarray(samples), np.asarray(atlas_rows), np.asarray(labels)
    if samples.ndim != 2 or samples.shape[1] != 4:
        raise ValueError("sample table must be [N, 4] (scan, x, y, z), got shape %s" % (samples.shape,))
    n = samples.shape[0]
    if atlas_rows.shape != (n, 15):
        raise ValueError("atlas rows must be [%d, 15] (one per sample), got shape %s" % (n, atlas_rows.shape))
    if labels.shape != (n,):
        raise ValueError("labels must be [%d] (one per sample), got shape %s" % (n, labels.shape))
    dims = np.asarray([tuple(int(d) for d in s) for s in shapes], dtype=np.int64).reshape(-1, 3)
    if n == 0:
        return
    scan = samples[:, 0].astype(np.int64)
    bad = np.nonzero((scan < 0) | (scan >= len(dims)))[0]
    if len(bad):
        raise ValueError("sample %d: scan index %d out of range [0, %d)" % (bad[0], scan[bad[0]], len(dims)))
    c = samples[:, 1:].astype(np.int64)
    bad = np.nonzero(((c < 0) | (c >= dims[scan])).any(1))[0]
    if len(bad):
        i = bad[0]
        raise ValueError("sample %d: centre %s outside scan %d of shape %s" % (i, tuple(c[i]), scan[i], tuple(dims[scan[i]])))


class ScanTrainingSet(object):
    """A training set held as its normalised scans plus one row per sample, all on the device: (scan, x, y, z), the
    15 atlas priors at the centre and the class label (0..14).  About 80 B per sample instead of the 12 KB of patches
    that generate_training_set materialises on the host; every minibatch is gathered from the scans by
    sc_gather_samples.  Row i is row i of what load_data + generate_training_set return for the same seeds.

        scans = load_scan_training_set(options)
        net.fit(scans)
        in1, in2, in3, in4, y = scans.gather(idx)       # CUDA tensors of rows idx
    """

    def __init__(self, volumes, samples, atlas_rows, labels, names=(), device=None):
        """volumes: float32 [X, Y, Z] per scan (numpy or CUDA tensors); samples int [N, 4]; atlas_rows [N, 15];
        labels [N].  The table is validated here, on the host, before any upload."""
        samples = np.ascontiguousarray(samples, dtype=np.int32)
        atlas_rows = np.ascontiguousarray(atlas_rows, dtype=np.float32)
        labels = np.ascontiguousarray(labels, dtype=np.uint8)
        for v in volumes:
            if len(v.shape) != 3:
                raise ValueError("scan volumes must be 3-D, got shape %s" % (tuple(v.shape),))
        check_sample_table([tuple(v.shape) for v in volumes], samples, atlas_rows, labels)
        import torch
        from . import parallel
        self.ctx = get_context(device)
        d = self.ctx.device
        self.volumes = [v.to('cuda:%d' % d, torch.float32).contiguous() if torch.is_tensor(v) else _dev(v, d, np.float32)
                        for v in volumes]
        self.table = self.ctx.scan_table(self.volumes)
        self.samples, self.atlas, self.labels = _dev(samples, d), _dev(atlas_rows, d), _dev(labels, d)
        self.y = labels                       # host copy: TrainSplit's stratified folds
        self.names = list(names)
        self.fingerprint = parallel.scan_set_fingerprint(samples, atlas_rows, labels, self.volumes)

    def __len__(self):
        return len(self.y)

    def device_bytes(self):
        """bytes of device memory the set holds"""
        ts = self.volumes + [self.table, self.samples, self.atlas, self.labels]
        return int(sum(t.numel() * t.element_size() for t in ts))

    def gather(self, idx=None, ctx=None):
        """-> (in1, in2, in3, in4, y): axial / coronal / saggital [n, 1, 32, 32] float32, atlas [n, 15] float32 and
        labels [n] uint8 CUDA tensors of rows idx (host integer array, CUDA int64 tensor, or None for every row).  A host
        idx is range-checked; a device idx is trusted.  ctx: the sc_ctx to launch on (default: the data layer's)."""
        import torch
        n = None
        if idx is None:
            n = len(self)
        elif not torch.is_tensor(idx):
            idx = np.ascontiguousarray(idx, dtype=np.int64).reshape(-1)
            if idx.size and (idx.min() < 0 or idx.max() >= len(self)):
                raise IndexError("row index out of range [0, %d)" % len(self))
            idx = _dev(idx, self.ctx.device)
        return (ctx or self.ctx).gather_samples(self.table, len(self.volumes), self.samples, self.atlas, self.labels,
                                                idx=idx, n=n)

    def to_arrays(self, chunk=32768):
        """(x_axial, x_cor, x_sag, x_atlas, y) host arrays: what generate_training_set returns for the same seeds."""
        n = len(self)
        out = [np.empty((n, 1, 32, 32), np.float32) for _ in range(3)] + [np.empty((n, 15), np.float32), np.empty(n, np.uint8)]
        for s in range(0, n, chunk):
            for o, t in zip(out, self.gather(np.arange(s, min(n, s + chunk)))):
                o[s:s + len(t)] = t.cpu().numpy()
        return tuple(out)


def load_scan_training_set(options, randomize=True, device=None):
    """load_data followed by generate_training_set, kept on the device -> ScanTrainingSet.

    Same semantics and the same random draws as the materialised path, so that the same ``random`` / ``np.random``
    seeds give the same set in the same order: per subject (sorted sub-folders of train_folder) the train-path
    normalised T1 (base.py:146), every voxel with label 1..14 in np.nonzero order and as many shuffled label-15 voxels
    (base.py:153-181), the atlas rows without background fix (quirk Q4), labels with 15 -> 0; subjects concatenated,
    then one permutation drawn as generate_training_set draws it.  Only the normalised T1 volumes stay on the device;
    the atlas rows and labels are picked from the host arrays the NIfTI reader returns (an upload of the 15-channel
    priors would move 60 B per voxel to read 60 B per sample)."""
    if tuple(options['patch_size']) != (32, 32):
        raise ValueError("only patch_size (32, 32) is implemented")
    ctx = get_context(options.get('device') if device is None else device)
    dir_name = options['train_folder']
    _register_folder(dir_name, options)
    subjects = [f for f in sorted(os.listdir(dir_name)) if os.path.isdir(os.path.join(dir_name, f))]
    names, vols, samples, atlas_rows, labels = [], [], [], [], []
    for k, subject in enumerate(subjects):
        image_name = os.path.join(dir_name, subject, options['t1_name'])
        atlas_name = os.path.join(dir_name, subject, 'tmp', 'MNI_sub_probabilities.nii.gz')
        _require_registered(atlas_name)
        vols.append(_dev(_train_normalise(load_nii(image_name).get_data()), ctx.device, np.float32))
        mask = load_nii(os.path.join(dir_name, subject, options['roi_name'])).get_data()
        cen = _training_centres(mask, ctx.device)
        x, y, z = cen[:, 0], cen[:, 1], cen[:, 2]
        lab = mask[x, y, z].astype(np.uint8)
        lab[lab == 15] = 0
        atlas_rows.append(np.asarray(load_nii(atlas_name).get_data()[x, y, z], dtype=np.float32))
        samples.append(np.concatenate([np.full((len(cen), 1), k, np.int32), cen], axis=1))
        labels.append(lab)
        names.append(image_name)
    samples = np.concatenate(samples) if samples else np.zeros((0, 4), np.int32)
    atlas_rows = np.concatenate(atlas_rows) if atlas_rows else np.zeros((0, 15), np.float32)
    labels = np.concatenate(labels) if labels else np.zeros(0, np.uint8)
    perm = _training_order(len(labels), randomize)
    if perm is not None:
        samples, atlas_rows, labels = samples[perm], atlas_rows[perm], labels[perm]
    if options.get('debug') == 'True':
        print("    --> X_TRAIN: ", len(labels), "samples from", len(vols), "scans")
    return ScanTrainingSet(vols, samples, atlas_rows, labels, names=names, device=ctx.device)
