"""ctypes binding of libsubcort_b200.so (the stub INTEGRATION.md shows).

PyTorch is used only as glue: device memory (torch tensors' ``data_ptr()``), the current
CUDA stream and, for multi-GPU training, ``torch.distributed``.  Every compute call goes
through the C-ABI declared in ``include/subcort_b200.h``.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libsubcort_b200.so")
PARAM_FLOATS = 883455
# sc_dtype codes of raw (un-normalised) volumes, include/subcort_b200.h
DTYPE_CODES = {"u1": 1, "i1": 2, "u2": 3, "i2": 4, "u4": 5, "i4": 6, "f4": 7, "f8": 8}

# sc_scan of include/subcort_b200.h: {const float* vol; int32_t dims[3]; int32_t reserved;}
SCAN_DTYPE = np.dtype([("vol", "<u8"), ("dims", "<i4", (3,)), ("reserved", "<i4")])
assert SCAN_DTYPE.itemsize == 24

# sc_structure_metrics of include/subcort_b200.h, one row per structure 1..14
METRICS_DTYPE = np.dtype([("n_seg", "<i8"), ("n_ref", "<i8"), ("n_both", "<i8"), ("dice", "<f8"), ("vol_seg_mm3", "<f8"),
                          ("vol_ref_mm3", "<f8"), ("hd_mm", "<f8"), ("hd95_mm", "<f8"), ("assd_mm", "<f8")])
assert METRICS_DTYPE.itemsize == 72

_lib = None


class NativeError(RuntimeError):
    pass


def _p(t):
    return ctypes.POINTER(t)


_c_f, _c_i32, _c_u8, _c_i64 = ctypes.c_float, ctypes.c_int32, ctypes.c_uint8, ctypes.c_int64
_vp = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/subcort_b200.h one to one
PROTOTYPES = {
    "sc_version": (ctypes.c_int, []),
    "sc_last_error": (ctypes.c_char_p, []),
    "sc_create": (ctypes.c_int, [ctypes.c_int, _p(_vp)]),
    "sc_destroy": (ctypes.c_int, [_vp]),
    "sc_set_option": (ctypes.c_int, [_vp, ctypes.c_char_p, _c_i64]),
    "sc_get_counter": (_c_i64, [_vp, ctypes.c_char_p]),
    "sc_profile_classes": (ctypes.c_int, []),
    "sc_profile_name": (ctypes.c_char_p, [ctypes.c_int]),
    "sc_profile_read": (ctypes.c_int, [_vp, _p(ctypes.c_double), _p(_c_i64), ctypes.c_int]),
    "sc_load_weights": (ctypes.c_int, [_vp, _vp, _c_i64]),
    "sc_get_params": (ctypes.c_int, [_vp, _vp, _c_i64]),
    "sc_nonzero_coords": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _p(_c_i32), _vp, _c_i64, _p(_c_i64), _vp]),
    "sc_dilate_mask": (ctypes.c_int, [_vp, _vp, _p(_c_i32), ctypes.c_int, _vp, _vp]),
    "sc_import_volume": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _p(_c_i32), ctypes.c_int, _vp, _vp]),
    "sc_upload_volume_box": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _p(_c_i32), ctypes.c_int, ctypes.c_int, _p(_c_i32), _vp, _vp, _vp]),
    "sc_normalise_volume": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _p(_c_i32), _vp, _p(ctypes.c_double), _vp]),
    "sc_candidate_mask": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _p(_c_i32), _vp, _vp]),
    "sc_mask_bbox": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _p(_c_i32), _p(_c_i64), _vp]),
    "sc_post_process": (ctypes.c_int, [_vp, _vp, _vp, _p(_c_i32), _vp, _vp]),
    "sc_evaluate_segmentation": (ctypes.c_int, [_vp, _vp, _vp, _p(_c_i32), _p(ctypes.c_double), _vp, _vp, _vp]),
    "sc_ffd_grid_dims": (ctypes.c_int, [_p(_c_i32), _p(_c_i32)]),
    "sc_register_affine": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _p(ctypes.c_double), _vp, _p(_c_i32), _p(ctypes.c_double), _p(ctypes.c_double), _vp]),
    "sc_register_ffd": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _p(ctypes.c_double), _vp, _p(_c_i32), _p(ctypes.c_double), _p(ctypes.c_double), _vp, _vp]),
    "sc_warp_volume": (ctypes.c_int, [_vp, _vp, _p(_c_i32), ctypes.c_int, _p(ctypes.c_double), _p(ctypes.c_double), _vp, _p(_c_i32),
                                      _p(ctypes.c_double), _vp, _vp]),
    "sc_register_objective": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _p(ctypes.c_double), _vp, _p(_c_i32), _p(ctypes.c_double),
                                             _p(ctypes.c_double), _vp, _p(ctypes.c_double), _vp, _vp, _vp]),
    "sc_prior_mask": (ctypes.c_int, [_vp, _vp, _p(_c_i32), ctypes.c_int, _vp, _vp]),
    "sc_gather_patches": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _vp, ctypes.c_int, _vp, _c_i64, _vp, _vp, _vp, _vp, _vp]),
    "sc_gather_center_labels": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _vp, _c_i64, _vp, _vp]),
    "sc_gather_samples": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp, _vp, _vp, _c_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sc_forward": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _vp, _vp, _vp]),
    "sc_forward_host": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _vp, _vp, _vp]),
    "sc_dense_layer": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _c_i64, _vp, ctypes.c_int, _vp]),
    "sc_forward_from_volume": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _vp, _vp, _c_i64, _vp, _vp, _vp]),
    "sc_segment_volume": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _vp, _p(_c_i32), _vp, _vp, _vp, _vp]),
    "sc_segment_volume_mc": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _vp, _p(_c_i32), _vp, ctypes.c_int, ctypes.c_uint64, _vp, _vp,
                                            _vp, _vp, _vp]),
    "sc_atlas_ready_event": (ctypes.c_int, [_vp, _vp]),
    "sc_segment_volume_host": (ctypes.c_int, [_vp, _vp, _p(_c_i32), _vp, _p(_c_i32), _vp, _vp, _vp, _vp]),
    "sc_scatter": (ctypes.c_int, [_vp, _vp, _c_i64, _vp, _vp, _p(_c_i32), _vp, _vp, _vp]),
    "sc_train_forward_backward": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, ctypes.c_uint64, _vp, _vp, _vp]),
    "sc_grad_buffer": (ctypes.c_int, [_vp, _p(_vp)]),
    "sc_param_buffer": (ctypes.c_int, [_vp, _p(_vp)]),
    "sc_adam_step": (ctypes.c_int, [_vp, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _vp]),
    "sc_reset_optimizer": (ctypes.c_int, [_vp]),
    "sc_fused_export": (ctypes.c_int, [_vp, _vp]),
    "sc_fused_attach": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp]),
    "sc_allreduce_adam_step": (ctypes.c_int, [_vp, _c_f, _c_f, _c_f, _c_f, _vp]),
    "sc_set_allreduce_hook": (ctypes.c_int, [_vp, _vp, _vp]),
    "sc_eval_batch": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _vp, _vp]),
}


def load_library():
    """dlopen the in-tree library; fail loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "%s is missing: build it with `python __graft_entry__.py` (or `make -C "
            "sub-cortical_segmentation_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _check(status):
    if status != 0:
        raise NativeError("subcort_b200 error %d: %s" % (status, load_library().sc_last_error().decode("utf-8", "replace")))


def _dims(shape):
    return (_c_i32 * 3)(*[int(s) for s in shape[:3]])


def _mat(m):
    """4x4 matrix -> row-major double[16]"""
    return (ctypes.c_double * 16)(*[float(v) for v in np.asarray(m, np.float64).reshape(16)])


def _ptr(t):
    """device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        assert t.flags["C_CONTIGUOUS"]
        return t.ctypes.data
    assert t.is_contiguous()
    return t.data_ptr()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


class Context(object):
    """One sc_ctx (one GPU).  Methods take torch CUDA tensors unless named *_host."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = _vp()
        _check(self.lib.sc_create(int(device), ctypes.byref(h)))
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.lib.sc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- options / counters ---------------------------------------------------------------
    def set_option(self, key, value):
        _check(self.lib.sc_set_option(self.h, key.encode(), int(value)))

    def counter(self, key):
        return int(self.lib.sc_get_counter(self.h, key.encode()))

    def profile_read(self):
        """{kernel class: (summed ms, launches)} since the last read (needs set_option('profile', 1))."""
        n = self.lib.sc_profile_classes()
        ms = (ctypes.c_double * n)()
        cnt = (_c_i64 * n)()
        _check(self.lib.sc_profile_read(self.h, ms, cnt, n))
        return {self.lib.sc_profile_name(i).decode(): (ms[i], int(cnt[i])) for i in range(n) if cnt[i]}

    # -- parameters -------------------------------------------------------------------------
    def load_weights(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.float32)
        _check(self.lib.sc_load_weights(self.h, blob.ctypes.data, blob.size))

    def get_params(self):
        out = np.empty(PARAM_FLOATS, np.float32)
        _check(self.lib.sc_get_params(self.h, out.ctypes.data, out.size))
        return out

    # -- data layer ---------------------------------------------------------------------------
    def nonzero_coords(self, vol):
        """vol: CUDA tensor [X,Y,Z] (uint8/bool or float32/int32) -> int32 CUDA tensor [N,3], C-order."""
        import torch
        eb = vol.element_size()
        n = _c_i64(0)
        _check(self.lib.sc_nonzero_coords(self.h, _ptr(vol), eb, _dims(vol.shape), None, 0, ctypes.byref(n), _stream()))
        xyz = torch.empty((n.value, 3), dtype=torch.int32, device=vol.device)
        if n.value:
            _check(self.lib.sc_nonzero_coords(self.h, _ptr(vol), eb, _dims(vol.shape), _ptr(xyz), n.value, None, _stream()))
        return xyz

    def dilate_mask(self, mask, iterations):
        """uint8 CUDA mask [X,Y,Z] -> scipy.ndimage.binary_dilation(mask, iterations=iterations) as uint8 0/1"""
        import torch
        out = torch.empty_like(mask)
        _check(self.lib.sc_dilate_mask(self.h, _ptr(mask), _dims(mask.shape), int(iterations), _ptr(out), _stream()))
        return out

    # -- scan preparation (device-resident head of load_patch_batch / test_scan) ------------------
    def upload_volume(self, arr, channels=1):
        """numpy volume [X,Y,Z(,C)] of any supported dtype and memory order -> (uint8 CUDA tensor holding the C-ordered
        bytes, dtype).  A Fortran-ordered array (what a NIfTI file holds) is uploaded as it lies in memory -- no host
        transposition -- and reordered on the device (sc_import_volume)."""
        import torch
        arr = np.asarray(arr)
        if arr.dtype == np.bool_:
            arr = arr.view(np.uint8)
        if arr.dtype.str[1:] not in DTYPE_CODES:
            raise NativeError("unsupported volume dtype %s" % arr.dtype)
        shape = tuple(int(s) for s in arr.shape[:3])
        dev = "cuda:%d" % self.device
        if arr.flags["C_CONTIGUOUS"]:
            return torch.from_numpy(arr.reshape(-1).view(np.uint8)).to(dev, non_blocking=True), arr.dtype
        if not arr.flags["F_CONTIGUOUS"]:
            arr = np.asfortranarray(arr)
        host = torch.from_numpy(arr.reshape(-1, order="F").view(np.uint8))
        raw = torch.empty(host.numel(), dtype=torch.uint8, device=dev)
        step = 64 << 20           # pieces of 64 MB: small copies of other streams (statistics, counts) slip in between them
        for o in range(0, host.numel(), step):
            raw[o:o + step].copy_(host[o:o + step], non_blocking=True)
        out = torch.empty_like(raw)
        _check(self.lib.sc_import_volume(self.h, _ptr(raw), arr.dtype.itemsize, _dims(shape), int(channels), _ptr(out), _stream()))
        return out, arr.dtype

    def upload_volume_box(self, arr, box, channels=1, out=None):
        """only the box (x0,x1,y0,y1,z0,z1) of a host volume [X,Y,Z(,C)] goes to the device (strided DMA, no host copy): ->
        C-ordered CUDA tensor of the array's dtype and FULL shape whose box region holds the data; the rest is uninitialised
        (or keeps the contents of `out`).  The crop path uploads the atlas priors this way (sc_upload_volume_box)."""
        import torch
        arr = np.asarray(arr)
        if arr.dtype.str[1:] not in DTYPE_CODES:
            raise NativeError("unsupported volume dtype %s" % arr.dtype)
        fortran = not arr.flags["C_CONTIGUOUS"]
        if fortran and not arr.flags["F_CONTIGUOUS"]:
            arr = np.asfortranarray(arr)
        shape = tuple(int(s) for s in arr.shape[:3])
        dev = "cuda:%d" % self.device
        tdt = torch.from_numpy(np.zeros(1, arr.dtype)).dtype
        full = shape + ((int(channels),) if arr.ndim == 4 else ())
        if out is None:
            out = torch.empty(full, dtype=tdt, device=dev)
        staging = None
        if fortran:
            n = shape[0] * (box[3] - box[2]) * (box[5] - box[4]) * int(channels)        # whole x rows (contiguous runs of the y range)
            staging = torch.empty(n, dtype=tdt, device=dev)
        _check(self.lib.sc_upload_volume_box(self.h, ctypes.c_void_p(arr.ctypes.data), arr.dtype.itemsize, _dims(shape), int(channels),
                                             1 if fortran else 0, (_c_i32 * 6)(*[int(b) for b in box]), _ptr(staging), _ptr(out), _stream()))
        return out

    def normalise_volume(self, raw, dtype, shape, want_volume=True):
        """C-ordered raw volume bytes on the device -> (float32 CUDA tensor [X,Y,Z], mean_nz, std_nz) == numpy's
        (image - image[nz].mean()) / image[nz].std() cast to float32, bit for bit (base.py:358)."""
        import torch
        out = torch.empty(tuple(shape), dtype=torch.float32, device=raw.device) if want_volume else None
        ms = (ctypes.c_double * 2)()
        _check(self.lib.sc_normalise_volume(self.h, _ptr(raw), DTYPE_CODES[np.dtype(dtype).str[1:]], _dims(shape), _ptr(out), ms, _stream()))
        return out, ms[0], ms[1]

    def candidate_mask(self, raw, dtype, shape):
        """raw != 0 as a uint8 CUDA mask [X,Y,Z] (base.py:372)"""
        import torch
        mask = torch.empty(tuple(shape), dtype=torch.uint8, device=raw.device)
        _check(self.lib.sc_candidate_mask(self.h, _ptr(raw), DTYPE_CODES[np.dtype(dtype).str[1:]], _dims(shape), _ptr(mask), _stream()))
        return mask

    def mask_bbox(self, mask):
        """(half-open box (x0,x1,y0,y1,z0,z1) or None, number of non-zero voxels) of a uint8 CUDA mask"""
        box = (_c_i32 * 6)()
        n = _c_i64(0)
        _check(self.lib.sc_mask_bbox(self.h, _ptr(mask), _dims(mask.shape), box, ctypes.byref(n), _stream()))
        return (tuple(int(b) for b in box) if n.value else None), int(n.value)

    def post_process(self, seg, mask):
        """uint8 CUDA label volume + uint8 CUDA mask [X,Y,Z] -> filtered uint8 label volume (base.py:460-480)"""
        import torch
        out = torch.empty_like(seg)
        _check(self.lib.sc_post_process(self.h, _ptr(seg), _ptr(mask), _dims(seg.shape), _ptr(out), _stream()))
        return out

    def evaluate_segmentation(self, seg, ref, spacing=(1.0, 1.0, 1.0), confusion=False):
        """uint8 CUDA label volumes seg / ref [X,Y,Z] (0..15, 15 = background) -> (METRICS_DTYPE [14]: row l - 1 holds
        structure l, confusion int64 [15, 15] [ref class][seg class] or None).  Synchronises (sc_evaluate_segmentation)."""
        if tuple(seg.shape) != tuple(ref.shape) or seg.dim() != 3:
            raise ValueError("seg and ref must be 3-D volumes of one shape, got %s and %s" % (tuple(seg.shape), tuple(ref.shape)))
        out = np.zeros(14, METRICS_DTYPE)
        conf = np.zeros((15, 15), np.int64) if confusion else None
        sp = (ctypes.c_double * 3)(*[float(s) for s in spacing])
        _check(self.lib.sc_evaluate_segmentation(self.h, _ptr(seg), _ptr(ref), _dims(seg.shape), sp, out.ctypes.data,
                                                 None if conf is None else conf.ctypes.data, _stream()))
        return out, conf

    # -- atlas registration (include/subcort_b200.h) -----------------------------------------------
    def ffd_grid_dims(self, ref_shape):
        g = (_c_i32 * 3)()
        _check(self.lib.sc_ffd_grid_dims(_dims(ref_shape), g))
        return tuple(int(v) for v in g)

    def register_affine(self, ref, ref_vox2mm, flo, flo_vox2mm):
        """float32 CUDA volumes: subject T1 (reference) and template T1 (floating), 4x4 voxel -> mm matrices -> the 4x4
        affine (subject mm -> template mm) as a numpy array.  Synchronises (sc_register_affine)."""
        out = (ctypes.c_double * 16)()
        _check(self.lib.sc_register_affine(self.h, _ptr(ref), _dims(ref.shape), _mat(ref_vox2mm), _ptr(flo), _dims(flo.shape),
                                           _mat(flo_vox2mm), out, _stream()))
        return np.array(out[:], np.float64).reshape(4, 4)

    def register_ffd(self, ref, ref_vox2mm, flo, flo_vox2mm, affine):
        """-> float32 CUDA control-point grid [gx, gy, gz, 3] (template mm) refining `affine` (sc_register_ffd)"""
        import torch
        grid = torch.empty(self.ffd_grid_dims(ref.shape) + (3,), dtype=torch.float32, device=ref.device)
        _check(self.lib.sc_register_ffd(self.h, _ptr(ref), _dims(ref.shape), _mat(ref_vox2mm), _ptr(flo), _dims(flo.shape),
                                        _mat(flo_vox2mm), _mat(affine), _ptr(grid), _stream()))
        return grid

    def warp_volume(self, flo, flo_vox2mm, affine, grid, ref_shape, ref_vox2mm, out=None):
        """float32 CUDA volume [X,Y,Z] or [X,Y,Z,15] on the template grid -> the same on the subject grid through phi
        (grid None: affine only), 0 outside (sc_warp_volume)"""
        import torch
        ch = 15 if flo.dim() == 4 else 1
        shape = tuple(int(s) for s in ref_shape[:3]) + ((15,) if ch == 15 else ())
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=flo.device)
        _check(self.lib.sc_warp_volume(self.h, _ptr(flo), _dims(flo.shape), ch, _mat(flo_vox2mm), _mat(affine), _ptr(grid),
                                       _dims(shape), _mat(ref_vox2mm), _ptr(out), _stream()))
        return out

    def register_objective(self, ref, ref_vox2mm, flo, flo_vox2mm, affine, grid=None, want_grad=False):
        """-> (NMI, BE, J, d NMI / d A [3, 4] or None, d J / d grid CUDA tensor or None) at full resolution"""
        import torch
        val = (ctypes.c_double * 3)()
        ga = (ctypes.c_double * 12)() if want_grad else None
        gg = torch.empty_like(grid) if want_grad and grid is not None else None
        _check(self.lib.sc_register_objective(self.h, _ptr(ref), _dims(ref.shape), _mat(ref_vox2mm), _ptr(flo), _dims(flo.shape),
                                              _mat(flo_vox2mm), _mat(affine), _ptr(grid), val, ga, _ptr(gg), _stream()))
        return val[0], val[1], val[2], (np.array(ga[:]).reshape(3, 4) if want_grad else None), gg

    def prior_mask(self, priors, iterations=5):
        """float32 CUDA priors [X,Y,Z,15] -> float32 0/1 mask: channels 0..12 summing to > 0, dilated (sc_prior_mask)"""
        import torch
        out = torch.empty(tuple(priors.shape[:3]), dtype=torch.float32, device=priors.device)
        _check(self.lib.sc_prior_mask(self.h, _ptr(priors), _dims(priors.shape), int(iterations), _ptr(out), _stream()))
        return out

    def gather_patches(self, vol, xyz, atlas=None, bg_fix=True, views=(True, True, True)):
        import torch
        n = xyz.shape[0]
        outs = [torch.empty((n, 1, 32, 32), dtype=torch.float32, device=vol.device) if v else None for v in views]
        at = torch.empty((n, 15), dtype=torch.float32, device=vol.device) if atlas is not None else None
        _check(self.lib.sc_gather_patches(self.h, _ptr(vol), _dims(vol.shape), _ptr(atlas), int(bool(bg_fix)), _ptr(xyz), n,
                                          _ptr(outs[0]), _ptr(outs[1]), _ptr(outs[2]), _ptr(at), _stream()))
        return outs[0], outs[1], outs[2], at

    def gather_center_labels(self, labels, xyz):
        import torch
        y = torch.empty((xyz.shape[0],), dtype=torch.uint8, device=labels.device)
        _check(self.lib.sc_gather_center_labels(self.h, _ptr(labels), _dims(labels.shape), _ptr(xyz), xyz.shape[0], _ptr(y), _stream()))
        return y

    def scan_table(self, volumes):
        """float32 CUDA volumes [X,Y,Z] -> the sc_scan array sc_gather_samples reads (uint8 CUDA tensor).  The table
        holds raw pointers: the volumes must outlive it."""
        import torch
        t = np.zeros(len(volumes), SCAN_DTYPE)
        for k, v in enumerate(volumes):
            assert v.dtype == torch.float32 and v.dim() == 3 and v.is_contiguous()
            t[k]["vol"], t[k]["dims"] = v.data_ptr(), tuple(v.shape)
        return torch.from_numpy(t.view(np.uint8)).to("cuda:%d" % self.device)

    def gather_samples(self, table, n_scans, samples, atlas_rows=None, labels=None, idx=None, n=None,
                       views=(True, True, True), want_atlas=True, want_y=True):
        """Rows idx (None: the first n rows) of a device sample table (int32 [N,4] scan, x, y, z) ->
        (axial, coronal, saggital [n,1,32,32] float32, atlas [n,15] float32, y [n] uint8); outputs not asked for, or
        whose source is None, are None (sc_gather_samples)."""
        import torch
        if n is None:
            n = idx.shape[0] if idx is not None else samples.shape[0]
        d = samples.device
        outs = [torch.empty((n, 1, 32, 32), dtype=torch.float32, device=d) if v else None for v in views]
        at = torch.empty((n, 15), dtype=torch.float32, device=d) if want_atlas and atlas_rows is not None else None
        y = torch.empty((n,), dtype=torch.uint8, device=d) if want_y and labels is not None else None
        _check(self.lib.sc_gather_samples(self.h, _ptr(table), int(n_scans), _ptr(samples), _ptr(atlas_rows), _ptr(labels),
                                          _ptr(idx), int(n), _ptr(outs[0]), _ptr(outs[1]), _ptr(outs[2]), _ptr(at), _ptr(y),
                                          _stream()))
        return outs[0], outs[1], outs[2], at, y

    # -- network ------------------------------------------------------------------------------
    def forward(self, in1, in2, in3, in4, want_proba=True, want_label=True):
        import torch
        n = in1.shape[0]
        proba = torch.empty((n, 15), dtype=torch.float32, device=in1.device) if want_proba else None
        label = torch.empty((n,), dtype=torch.int32, device=in1.device) if want_label else None
        _check(self.lib.sc_forward(self.h, _ptr(in1), _ptr(in2), _ptr(in3), _ptr(in4), n, _ptr(proba), _ptr(label), _stream()))
        return proba, label

    def forward_host(self, in1, in2, in3, in4, want_proba=True, want_label=True):
        n = in1.shape[0]
        proba = np.empty((n, 15), np.float32) if want_proba else None
        label = np.empty((n,), np.int32) if want_label else None
        _check(self.lib.sc_forward_host(self.h, _ptr(in1), _ptr(in2), _ptr(in3), _ptr(in4), n, _ptr(proba), _ptr(label), _stream()))
        return proba, label

    def dense_layer(self, which, x, backend):
        """one head layer on its own: which 0..2 = d1 of a branch, 3 = FC1, 4 = fc_2 (see subcort_b200.h)"""
        import torch
        width = {0: 192, 1: 192, 2: 192, 3: 576, 4: 272}[which]
        out = torch.zeros((x.shape[0], width), dtype=torch.float32, device=x.device)
        _check(self.lib.sc_dense_layer(self.h, which, _ptr(x), x.shape[0], _ptr(out), backend, _stream()))
        return out

    def forward_from_volume(self, vol, atlas, xyz, want_proba=True, want_label=True):
        import torch
        n = xyz.shape[0]
        proba = torch.empty((n, 15), dtype=torch.float32, device=vol.device) if want_proba else None
        label = torch.empty((n,), dtype=torch.int32, device=vol.device) if want_label else None
        _check(self.lib.sc_forward_from_volume(self.h, _ptr(vol), _dims(vol.shape), _ptr(atlas), _ptr(xyz), n,
                                               _ptr(proba), _ptr(label), _stream()))
        return proba, label

    def segment_volume(self, vol, atlas, box=None, cand_mask=None, label_vol=None, proba_vol=None, atlas_ready=None):
        """atlas_ready: a torch.cuda.Event recorded behind an upload of `atlas` on another stream; the call waits for it
        only when the FC head first reads the priors, so the upload overlaps the convolution phase."""
        cbox = (_c_i32 * 6)(*[int(b) for b in box]) if box is not None else None
        if atlas_ready is not None:
            _check(self.lib.sc_atlas_ready_event(self.h, atlas_ready.cuda_event))
        _check(self.lib.sc_segment_volume(self.h, _ptr(vol), _dims(vol.shape), _ptr(atlas), cbox, _ptr(cand_mask),
                                          _ptr(label_vol), _ptr(proba_vol), _stream()))

    def segment_volume_mc(self, vol, atlas, samples, seed=0, box=None, cand_mask=None, label_vol=None, proba_vol=None,
                          entropy_vol=None, mi_vol=None, atlas_ready=None):
        """Monte-Carlo dropout over segment_volume (sc_segment_volume_mc): `samples` passes of the FC head with the training
        dropout masks drawn from `seed`; writes the arg-max and the mean of the passes' softmax, its entropy (nats) and the
        mutual information into whichever of the four CUDA volumes are given, at the voxels segment_volume writes."""
        cbox = (_c_i32 * 6)(*[int(b) for b in box]) if box is not None else None
        if atlas_ready is not None:
            _check(self.lib.sc_atlas_ready_event(self.h, atlas_ready.cuda_event))
        _check(self.lib.sc_segment_volume_mc(self.h, _ptr(vol), _dims(vol.shape), _ptr(atlas), cbox, _ptr(cand_mask), int(samples),
                                             int(seed), _ptr(label_vol), _ptr(proba_vol), _ptr(entropy_vol), _ptr(mi_vol), _stream()))

    def segment_volume_host(self, vol, atlas, box=None, cand_mask=None, want_proba=False, label_out=None):
        """numpy (or pinned torch CPU) in -> numpy uint8 label volume (+ float32 proba volume)."""
        shape = tuple(int(s) for s in vol.shape[:3])
        label = label_out if label_out is not None else np.zeros(shape, np.uint8)
        proba = np.zeros(shape + (15,), np.float32) if want_proba else None
        cbox = (_c_i32 * 6)(*[int(b) for b in box]) if box is not None else None
        _check(self.lib.sc_segment_volume_host(self.h, _ptr(vol), _dims(shape), _ptr(atlas), cbox, _ptr(cand_mask),
                                               _ptr(label), _ptr(proba), _stream()))
        return label, proba

    def scatter(self, xyz, dims, label=None, proba=None, label_vol=None, proba_vol=None):
        _check(self.lib.sc_scatter(self.h, _ptr(xyz), xyz.shape[0], _ptr(label), _ptr(proba), _dims(dims),
                                   _ptr(label_vol), _ptr(proba_vol), _stream()))

    # -- training -----------------------------------------------------------------------------
    def train_forward_backward(self, in1, in2, in3, in4, y, n_global=None, seed=0, drop_masks=None, loss_out=None):
        import torch
        n = in1.shape[0]
        loss = loss_out if loss_out is not None else torch.zeros(1, dtype=torch.float32, device=in1.device)
        _check(self.lib.sc_train_forward_backward(self.h, _ptr(in1), _ptr(in2), _ptr(in3), _ptr(in4), _ptr(y), n,
                                                  int(n_global or n), int(seed), _ptr(drop_masks), _ptr(loss), _stream()))
        return loss

    def _buffer(self, fn):
        import torch
        p = _vp()
        _check(fn(self.h, ctypes.byref(p)))
        return p.value

    def grad_tensor(self):
        """torch view (no copy) of the flat gradient buffer, for torch.distributed.all_reduce."""
        return _as_tensor(self._buffer(self.lib.sc_grad_buffer), PARAM_FLOATS, self.device)

    def param_tensor(self):
        return _as_tensor(self._buffer(self.lib.sc_param_buffer), PARAM_FLOATS, self.device)

    def adam_step(self, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0, stat_scale=1.0):
        _check(self.lib.sc_adam_step(self.h, lr, beta1, beta2, eps, grad_scale, stat_scale, _stream()))

    def set_sync_bn(self, enable=True):
        """Synchronised BatchNorm for data-parallel training: the BN reduction buffers are all-reduced over the ranks of
        torch.distributed's default group (sc_set_allreduce_hook), so that N ranks reproduce the single-device step on the
        same global batch.  Off (default): per-GPU batch statistics."""
        if not enable:
            _check(self.lib.sc_set_allreduce_hook(self.h, None, None))
            self._ar_cb = None
            return
        import torch
        import torch.distributed as dist
        device = self.device

        def hook(user, ptr, count, stream):
            try:
                t = torch.as_tensor(_CudaArrayHolder(ptr, int(count), "<f8"), device="cuda:%d" % device)
                # the library's stream: torch's default stream object when it is the legacy stream (wrapping handle 0 in an
                # ExternalStream does not order reliably against it)
                cur = torch.cuda.ExternalStream(stream, device=device) if stream else torch.cuda.default_stream(device)
                with torch.cuda.stream(cur):
                    if dist.get_backend() == "nccl":
                        dist.all_reduce(t)
                    else:                      # gloo reduces host tensors
                        h = t.cpu()
                        if os.environ.get("SC_DEBUG_HOOK"):
                            before = (float(h[0]), float(h[1]), float(h[192]))
                        dist.all_reduce(h)
                        t.copy_(h)
                        if os.environ.get("SC_DEBUG_HOOK"):
                            import sys
                            sys.stderr.write("hook rank %d stream %s: %r -> %r\n" % (dist.get_rank(), stream, before, (float(h[0]), float(h[1]), float(h[192]))))
                return 0
            except Exception:                  # never let an exception cross the C boundary
                import traceback
                traceback.print_exc()
                return -1

        self._ar_cb = ctypes.CFUNCTYPE(ctypes.c_int, _vp, _vp, _c_i64, _vp)(hook)
        _check(self.lib.sc_set_allreduce_hook(self.h, ctypes.cast(self._ar_cb, _vp), None))

    def fused_attach(self):
        """Exchange the CUDA IPC handles of the gradient / parameter / flag buffers over torch.distributed's default group and
        open the peers' buffers: afterwards allreduce_adam_step() replaces all_reduce + adam_step (one kernel over NVLink)."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        mine = np.zeros(192, np.uint8)
        _check(self.lib.sc_fused_export(self.h, mine.ctypes.data))
        if dist.get_backend() == "nccl":
            t = torch.from_numpy(mine).to("cuda:%d" % self.device)
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            allh = np.concatenate([p.cpu().numpy() for p in parts])
        else:
            t = torch.from_numpy(mine)
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            allh = np.concatenate([p.numpy() for p in parts])
        allh = np.ascontiguousarray(allh, dtype=np.uint8)
        _check(self.lib.sc_fused_attach(self.h, rank, world, allh.ctypes.data))
        dist.barrier()

    def allreduce_adam_step(self, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8):
        _check(self.lib.sc_allreduce_adam_step(self.h, lr, beta1, beta2, eps, _stream()))

    def reset_optimizer(self):
        _check(self.lib.sc_reset_optimizer(self.h))

    def eval_batch(self, in1, in2, in3, in4, y):
        import torch
        out = torch.zeros(2, dtype=torch.float32, device=in1.device)
        _check(self.lib.sc_eval_batch(self.h, _ptr(in1), _ptr(in2), _ptr(in3), _ptr(in4), _ptr(y), in1.shape[0], _ptr(out), _stream()))
        return out


class _CudaArrayHolder(object):
    def __init__(self, ptr, n, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def _as_tensor(ptr, n, device):
    import torch
    return torch.as_tensor(_CudaArrayHolder(ptr, n), device="cuda:%d" % device)
