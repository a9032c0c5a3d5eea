/* subcort_b200 -- C-ABI of the B200-native voxelwise hot path.
 *
 * The reference (sergivalverde/sub-cortical_segmentation) has NO FFI of its own: its
 * native arithmetic is generated at run time by Theano behind nolearn's NeuralNet
 * (cnn_cort/nets.py:233-246) and its data layer is numpy (cnn_cort/base.py).  Each entry
 * point below therefore names the reference *Python* interface it replaces; the
 * Python-side binding a maintainer adds is the ctypes stub shown in INTEGRATION.md
 * (implemented in sub-cortical_segmentation_b200/cnn_cort/_native.py).
 *
 * Conventions: extern "C"; plain pointers and sizes; every call returns 0 on success or
 * a negative sc_status, with a human-readable message in sc_last_error() (thread-local);
 * no exceptions cross the boundary.  Pointers named *_dev are CUDA device pointers on the
 * context's device (e.g. torch tensors' data_ptr()); *_host are host pointers (pinned
 * memory makes the copies asynchronous).  `stream` is a cudaStream_t passed as void*
 * (NULL = legacy default stream).  One sc_ctx per device per thread; contexts are
 * independent.  There is no CPU fallback: without a CUDA device sc_create fails.
 *
 * Coordinates are (x, y, z) int32 triples, volumes are C-ordered [X][Y][Z] (z fastest),
 * the atlas is [X][Y][Z][15] float32 -- the layouts cnn_cort/base.py uses after nibabel.
 */
#ifndef SUBCORT_B200_H
#define SUBCORT_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define SC_API __attribute__((visibility("default")))
#else
#define SC_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sc_ctx sc_ctx;

typedef enum {
  SC_OK = 0,
  SC_ERR_CUDA = -1,        /* a CUDA runtime/driver call failed */
  SC_ERR_ARG = -2,         /* bad argument (null pointer, negative size, unsupported patch size ...) */
  SC_ERR_STATE = -3,       /* call order violated (e.g. forward before sc_load_weights) */
  SC_ERR_NOMEM = -4,       /* device workspace could not be allocated */
  SC_ERR_UNSUPPORTED = -5  /* device is not sm_100 */
} sc_status;

#define SC_NUM_CLASSES 15
#define SC_PATCH 32
#define SC_PARAM_FLOATS 883455   /* floats in nets/<name>/<name>.pkl, pickle order */
#define SC_NUM_ARRAYS 107        /* non-empty arrays in that pickle */

/* ---- context ------------------------------------------------------------------------ */
SC_API int sc_version(void);
SC_API const char* sc_last_error(void);
/* replaces: THEANO_FLAGS device selection, cnn_cort/load_options.py:54-57 */
SC_API int sc_create(int device, sc_ctx** out);
SC_API int sc_destroy(sc_ctx* ctx);
/* knobs: "gemm" = 1 tcgen05 bf16x3 (the product path, always the default: sc_create fails where it cannot be brought up)
 *        | 0 exact-fp32 SIMT kernels (cross-check back-end for the parity tests only);
 *        "chunk_voxels" = voxels per head chunk in sc_segment_volume; "profile" = 0 | 1;
 *        "tc_compact" 0 | 1 (candidate-row compaction of the FC head, default 1), "gather_ctas_per_sm" 0..32,
 *        "tc_timing" = kernel class whose launches record per-role wait cycles (debug). */
SC_API int sc_set_option(sc_ctx* ctx, const char* key, int64_t value);
SC_API int64_t sc_get_counter(sc_ctx* ctx, const char* key); /* "launches": kernels launched so far */
/* per-kernel-class device times: after sc_set_option(ctx, "profile", 1) every launch is bracketed by
 * CUDA events on its stream; sc_profile_read synchronises, returns summed ms and launch counts per
 * class (arrays of at least sc_profile_classes() entries) and resets the accumulators. */
SC_API int sc_profile_classes(void);
SC_API const char* sc_profile_name(int cls);
SC_API int sc_profile_read(sc_ctx* ctx, double* ms_out, int64_t* launches_out, int n);

/* ---- parameters ----------------------------------------------------------------------
 * replaces: nolearn NeuralNet.load_params_from / save_params_to (call site nets.py:251).
 * `blob_host` is the concatenation of the 107 arrays of the OrderedDict in pickle order
 * (SC_PARAM_FLOATS floats).  The library keeps that master copy on the device and derives
 * the inference layouts (filter flip for flip_filters=True, BN folded to scale/shift,
 * transposed / padded / split-bf16 GEMM operands). */
SC_API int sc_load_weights(sc_ctx* ctx, const float* blob_host, int64_t n_floats);
SC_API int sc_get_params(sc_ctx* ctx, float* blob_host, int64_t n_floats);

/* ---- candidate voxels ----------------------------------------------------------------
 * replaces: get_mask_voxels(mask) cnn_cort/base.py:310-331 (np.nonzero order, C-order).
 * elem_bytes: 1 (uint8/bool mask) or 4 (float32/int32 image, tested != 0).
 * Writes up to `capacity` triples; *n_out_host receives the total count (synchronises). */
SC_API int sc_nonzero_coords(sc_ctx* ctx, const void* vol_dev, int elem_bytes, const int32_t dims[3],
                      int32_t* xyz_dev, int64_t capacity, int64_t* n_out_host, void* stream);

/* replaces: scipy.ndimage.binary_dilation(mask, iterations=10) of the crop path (base.py:369): default
 * 6-connected structuring element, zero border.  mask/out uint8 [X][Y][Z] (0 / non-zero in, 0 / 1 out), out != mask. */
SC_API int sc_dilate_mask(sc_ctx* ctx, const uint8_t* mask_dev, const int32_t dims[3], int iterations,
                   uint8_t* out_dev, void* stream);

/* ---- scan preparation on the device ---------------------------------------------------
 * replaces: the host-side head of load_patch_batch / test_scan (base.py:357-372).  A scan is uploaded once in the
 * array order the NIfTI file has; everything up to the label volume stays on the device. */
typedef enum { SC_DT_U8 = 1, SC_DT_I8, SC_DT_U16, SC_DT_I16, SC_DT_U32, SC_DT_I32, SC_DT_F32, SC_DT_F64 } sc_dtype;
/* NIfTI (Fortran) order -> the C order used everywhere else: src is [channels][Z][Y][X] (x fastest, what nibabel's
 * get_data() holds in memory), dst is [X][Y][Z][channels]; bit-preserving for elements of 1, 2, 4 or 8 bytes. */
SC_API int sc_import_volume(sc_ctx* ctx, const void* src_dev, int elem_bytes, const int32_t dims[3], int channels,
                     void* dst_dev, void* stream);
/* Crop mode (base.py:367-369): the atlas priors are only read at the candidate voxels, so only the candidates' bounding
 * box {x0,x1,y0,y1,z0,z1} of the HOST array (94 % of a scan's bytes are priors) is uploaded: strided DMA copies into
 * staging_dev (Fortran-ordered source: >= X * box_y * box_z * channels * elem_bytes bytes -- whole x rows are moved, the
 * x range is cut on the device; NULL for a C-ordered source) and a
 * reorder into the box region of dst_dev, the full-size C-ordered [X][Y][Z][channels] device volume.  Voxels outside
 * the box keep whatever dst_dev held.  src_host should be page-locked (pageable memory makes the copies synchronous). */
SC_API int sc_upload_volume_box(sc_ctx* ctx, const void* src_host, int elem_bytes, const int32_t dims[3], int channels,
                         int fortran_order, const int32_t box[6], void* staging_dev, void* dst_dev, void* stream);
/* replaces: image_norm = (image - image[np.nonzero(image)].mean()) / image[np.nonzero(image)].std() (base.py:358),
 * cast to float32 as the patches are (base.py:383).  numpy's result bit for bit: same dtype promotion, same pairwise
 * summation order (csrc/prep.cu).  vol_dev: C-ordered raw volume of `dtype`; out_dev float32 (NULL: statistics only);
 * mean_std_host (nullable): the two scalars.  Synchronises the stream. */
SC_API int sc_normalise_volume(sc_ctx* ctx, const void* vol_dev, int dtype, const int32_t dims[3], float* out_dev,
                        double* mean_std_host, void* stream);
/* replaces: image.astype('bool') (base.py:372) / the truth value scipy's binary_dilation takes of the registered mask
 * (base.py:369): mask_dev[v] = vol[v] != 0 as uint8. */
SC_API int sc_candidate_mask(sc_ctx* ctx, const void* vol_dev, int dtype, const int32_t dims[3], uint8_t* mask_dev, void* stream);
/* half-open bounding box {x0,x1,y0,y1,z0,z1} and number of the non-zero voxels of a uint8 mask (all zeros when empty):
 * the box sc_segment_volume restricts its convolutions to.  Synchronises the stream. */
SC_API int sc_mask_bbox(sc_ctx* ctx, const uint8_t* mask_dev, const int32_t dims[3], int32_t box_host[6],
                 int64_t* count_host, void* stream);

/* ---- orthogonal patch gather ---------------------------------------------------------
 * replaces: get_patches x3 views (base.py:272-308) + the atlas vector with background fix
 * (base.py:387-394) of one load_patch_batch batch.  Outputs are [n][1][32][32] float32 per
 * view and [n][15] float32; any output pointer may be NULL to skip it.  bg_fix=1 applies
 * "row sums to 0 -> row[14] = 1" (test path); 0 leaves rows untouched (train path, Q4). */
SC_API int sc_gather_patches(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3],
                      const float* atlas_dev, int bg_fix, const int32_t* xyz_dev, int64_t n,
                      float* axial_dev, float* coronal_dev, float* saggital_dev,
                      float* atlas_out_dev, void* stream);
/* the same windows of an integer label volume (load_patch_vectors, base.py:156-160);
 * only the centre pixel is ever consumed (base.py:85), so this returns labels[n] uint8. */
SC_API int sc_gather_center_labels(sc_ctx* ctx, const uint8_t* labels_dev, const int32_t dims[3],
                            const int32_t* xyz_dev, int64_t n, uint8_t* y_dev, void* stream);

/* ---- training minibatch from device-resident scans -----------------------------------
 * replaces: the patch arrays of load_patch_vectors / generate_training_set (base.py:53-184), i.e.
 * 12 KB of materialised patches per training sample, by a per-minibatch gather from the scans.
 * A training set is a table of N sample rows (scan, x, y, z) int32 [N][4] (16-byte aligned) over
 * n_scans caller-owned float32 volumes [X][Y][Z] (C order, normalised), optionally with an atlas
 * row float32 [N][15] and a label uint8 [N] per sample.  For i < n the call writes row
 * r = idx_dev[i] (r = i when idx_dev is NULL) of the table: the axial / coronal / saggital
 * patches [n][1][32][32] of scan `scan` around (x, y, z), exactly get_patches's windows and zero
 * fill (base.py:272-308), atlas_out[i] = atlas_rows[r] and y_out[i] = labels[r].  Any output may be
 * NULL; n == 0 is a no-op.  SC_ERR_ARG: negative counts, a NULL table or scan list (n > 0), an
 * atlas / label output requested without its source.
 * The table is device data and is not range-checked on the device: the caller guarantees
 * 0 <= idx[i] < N, 0 <= scan < n_scans, and a centre inside its scan's dims (cnn_cort checks
 * the table once, when the set is built).  A scan index outside [0, n_scans) yields zero
 * patches rather than an out-of-bounds read. */
typedef struct { const float* vol; int32_t dims[3]; int32_t reserved; } sc_scan;   /* 24 bytes; vol: caller-owned device array */
SC_API int sc_gather_samples(sc_ctx* ctx, const sc_scan* scans_dev, int n_scans, const int32_t* samples_dev,
                      const float* atlas_rows_dev, const uint8_t* labels_dev, const int64_t* idx_dev, int64_t n,
                      float* axial_dev, float* coronal_dev, float* saggital_dev, float* atlas_out_dev,
                      uint8_t* y_out_dev, void* stream);
/* Training-time augmentation in the same gather: every sample's three patches are resampled through one random 3-D similarity
 * about its centre voxel, then given a random contrast, brightness and Gaussian noise.  Arguments, outputs, NULL rules and trust
 * rules are those of sc_gather_samples; atlas_out and y_out are its rows unchanged, which stays correct because the transform
 * keeps the centre voxel fixed.
 *   Random numbers are keyed by (seed, epoch, table row r = idx[i]), never by the batch position i, so a shuffled minibatch, a
 *   validation fold or a data-parallel shard sees the same transform for the same row: with s_e = seed ^ (epoch *
 *   0xD1B54A32D192ED03) (uint64, wrapping) and u(k) = (hash3(s_e, r * 8192 + k) + 0.5) * 2^-32 in (0, 1) (hash3 of
 *   csrc/common.cuh):
 *     rotation axis  k = (sqrt(1 - z^2) cos(2 pi u(1)), sqrt(1 - z^2) sin(2 pi u(1)), z), z = 2 u(0) - 1 (uniform on the sphere);
 *     angle          theta = rotation_deg * (2 u(2) - 1) degrees;          scale  s = (1 + scale)^(2 u(3) - 1);
 *     contrast       a = 1 + intensity * (2 u(4) - 1);                     brightness  b = intensity * (2 u(5) - 1);
 *     noise          pixel (view v, row i, column j): g = sqrt(-2 ln u(n)) cos(2 pi u(n + 1)), n = 1024 + 2 (v * 1024 + i * 32 + j).
 *   Geometry: M = s R(k, theta), R by Rodrigues' formula, evaluated in double and rounded to float per entry.  Pixel (i, j) of a
 *   view sits at the voxel-index offset o = (i - 16) e_row + (j - 16) e_col from the centre c, with the axes of get_patches
 *   (axial: rows x, columns y; coronal: rows x, columns z; saggital: rows y, columns z), and samples the scan at
 *   p = c + (i - 16) M e_row + (j - 16) M e_col (float).  The transform acts in voxel-index space, which is isotropic in mm
 *   when the scans are on the [model] resample_mm grid.
 *   Value: trilinear interpolation at p of the zero-extended volume (a corner voxel outside the scan contributes 0: the
 *   continuous form of get_patches's zero fill), float accumulation in a fixed corner order; out = a * value + b + noise * g for
 *   every pixel, the zero fill included.  No atomics: the same arguments give byte-identical outputs.
 *   With all four ranges 0 the outputs equal those of sc_gather_samples: M = I exactly, p is the integer voxel, a = 1, b = 0.
 *   No mirroring: the 14 structures are seven left / right pairs (Kushibar et al. 2018), and a mirrored patch would need its
 *   label and its prior channels swapped to the other side's; that is not done here.
 * SC_ERR_ARG, outputs untouched, in addition to the checks of sc_gather_samples: aug NULL, a non-finite range, rotation_deg
 * outside [0, 180], scale or noise below 0, intensity outside [0, 1).  The message names the entry point and the field. */
typedef struct {
  float rotation_deg;   /* max rotation angle in degrees, [0, 180] */
  float scale;          /* isotropic scale range sigma_s >= 0: s in [1 / (1 + sigma_s), 1 + sigma_s] */
  float intensity;      /* contrast / brightness range sigma_i in [0, 1) */
  float noise;          /* std of the additive Gaussian noise, >= 0 (normalised intensity units) */
  uint64_t seed;
  int64_t epoch;
} sc_augment;           /* 32 bytes */
SC_API int sc_gather_samples_augmented(sc_ctx* ctx, const sc_scan* scans_dev, int n_scans, const int32_t* samples_dev,
                                       const float* atlas_rows_dev, const uint8_t* labels_dev, const int64_t* idx_dev, int64_t n,
                                       const sc_augment* aug, float* axial_dev, float* coronal_dev, float* saggital_dev,
                                       float* atlas_out_dev, uint8_t* y_out_dev, void* stream);

/* ---- network forward (patchwise) -----------------------------------------------------
 * replaces: net.predict_proba / net.predict on {'in1','in2','in3','in4'}
 * (call sites base.py:425-428, 435-438).  proba_dev [n][15] and/or label_dev [n] may be
 * NULL.  Deterministic mode (stored BN statistics, no dropout). */
SC_API int sc_forward(sc_ctx* ctx, const float* in1_dev, const float* in2_dev, const float* in3_dev,
               const float* in4_dev, int64_t n, float* proba_dev, int32_t* label_dev, void* stream);
/* host-buffer form of the same call: H2D of the four inputs and D2H of the results inside. */
SC_API int sc_forward_host(sc_ctx* ctx, const float* in1_host, const float* in2_host, const float* in3_host,
                    const float* in4_host, int64_t n, float* proba_host, int32_t* label_host, void* stream);
/* gather + forward without materialising patches on the host: one test_scan batch
 * (base.py:421-428) from a device-resident volume. */
SC_API int sc_forward_from_volume(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3],
                           const float* atlas_dev, const int32_t* xyz_dev, int64_t n,
                           float* proba_dev, int32_t* label_dev, void* stream);

/* one dense layer of the head on its own (parity tests of the GEMM back-ends): which = 0..2 the
 * d1 layer of the axial / coronal / saggital branch (in [n][576] flattened conv5 maps, 540 used -> out [n][192],
 * columns 0..179 valid), 3 = FC1 (in [n][576] = the feature buffer, 192 columns per view of which 180 are used -> out [n][576], columns 0..539 valid), 4 = fc_2
 * (in [n][576] = FC1 output | atlas | zero pad -> out [n][272]).  backend: 0 SIMT fp32, 1 tcgen05 split-bf16 (three MMAs).
 * replaces: DenseLayer + PReLU, cnn_cort/nets.py:179-180, 217-218, 227-228. */
SC_API int sc_dense_layer(sc_ctx* ctx, int which, const float* in_dev, int64_t n, float* out_dev, int backend, void* stream);

/* ---- whole-volume inference (dense dilated formulation) -----------------------------
 * replaces: the body of test_scan (base.py:421-440) when the candidates are (nearly) all
 * voxels of a box: per view the branch runs as dilated convolutions over whole slices,
 * which is exactly the patchwise network evaluated at every pixel (DESIGN.md).
 * box = {x0,x1,y0,y1,z0,z1} half-open (NULL = whole volume).  cand_mask_dev (uint8
 * [X][Y][Z], NULL = every voxel of the box) selects which voxels are written; the others
 * keep whatever label_vol/proba_vol held.  label_vol_dev uint8 [X][Y][Z];
 * proba_vol_dev float32 [X][Y][Z][15] or NULL. */
SC_API int sc_segment_volume(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3],
                      const float* atlas_dev, const int32_t* box, const uint8_t* cand_mask_dev,
                      uint8_t* label_vol_dev, float* proba_vol_dev, void* stream);
/* The atlas priors are first read after the convolution phase.  A caller that uploads them on a side stream passes the
 * cudaEvent_t recorded behind that upload here; the NEXT sc_segment_volume call makes its stream wait for the event right
 * before the FC head instead of the caller serialising upload and convolutions.  One-shot (cleared by that call). */
SC_API int sc_atlas_ready_event(sc_ctx* ctx, void* cuda_event);
/* Monte-Carlo dropout (Gal & Ghahramani 2016) over the same computation: `samples` (T) stochastic passes of the FC head
 * with the dropout of training (p = 0.5, kept units x2) at *_l1drop, f1_drop and f2_drop; the convolutions run once.
 * Pass t (0 <= t < T) keeps unit j of [3][540] l1drop (k = c*9 + h*3 + w) | [540] f1_drop | [540] f2_drop when
 * hash3(seed, t * 2700 + j) & 1 (the training step's mask of sample t, csrc/common.cuh), ONE mask for every voxel; that
 * is the deterministic head with the weight rows of the dropped inputs zeroed and the kept ones doubled.  Per voxel,
 * with p_t the softmax of pass t (atlas background fix as above):
 *   proba_vol   p = (1/T) sum_t p_t, float32 [X][Y][Z][15];   label_vol  the first arg-max of p, uint8 [X][Y][Z];
 *   entropy_vol H = -sum_c p_c ln p_c in nats (0 ln 0 = 0), float32 [X][Y][Z];
 *   mi_vol      max(0, H - (1/T) sum_t H(p_t)), the mutual information between prediction and weights (exactly 0 for T = 1).
 * Outputs are written exactly where sc_segment_volume writes (the candidates inside the box); any may be NULL, not all.
 * Deterministic: the same inputs and seed give byte-identical outputs.  sc_atlas_ready_event applies as above.
 * SC_ERR_ARG, outputs untouched: samples outside [1, 1024], the SIMT back-end selected ("gemm" = 0), NULL inputs or
 * all outputs NULL, bad dims, a box outside the volume.  The message names the argument. */
SC_API int sc_segment_volume_mc(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3], const float* atlas_dev,
                                const int32_t* box, const uint8_t* cand_mask_dev, int samples, uint64_t seed,
                                uint8_t* label_vol_dev, float* proba_vol_dev, float* entropy_vol_dev, float* mi_vol_dev,
                                void* stream);
/* host-buffer form: copies volume + atlas (+mask) in and the label (+proba) volume out. */
SC_API int sc_segment_volume_host(sc_ctx* ctx, const float* vol_host, const int32_t dims[3],
                           const float* atlas_host, const int32_t* box, const uint8_t* cand_mask_host,
                           uint8_t* label_vol_host, float* proba_vol_host, void* stream);

/* ---- post-processing ------------------------------------------------------------------
 * replaces: post_process_segmentation (base.py:460-480): per class 1..14 keep the 6-connected component that overlaps the
 * registered sub-cortical mask most (first maximum in scipy.ndimage.label's raster order; the reference's argmax == 0
 * quirk included, see csrc/postproc.cu).  seg / mask / out: uint8 [X][Y][Z]; mask non-zero = inside; out != seg. */
SC_API int sc_post_process(sc_ctx* ctx, const uint8_t* seg_dev, const uint8_t* mask_dev, const int32_t dims[3],
                    uint8_t* out_dev, void* stream);

/* ---- evaluation against manual labels --------------------------------------------------
 * replaces: the scipy / medpy-style host evaluation of a segmentation (binary_erosion surfaces, distance_transform_edt
 * per structure and direction, np.percentile); the reference has none.  seg / ref: uint8 [X][Y][Z] label volumes with
 * values 0..15, 15 counted as background (0) in both (as training does); seg_dev == ref_dev is allowed.  spacing: voxel
 * size in mm along x, y, z (finite, > 0).  For each structure l = 1..14 (metrics_host[l - 1]), A = (seg == l),
 * B = (ref == l): n_seg = |A|, n_ref = |B|, n_both = |A & B|; dice = 2 n_both / (n_seg + n_ref) (NaN when both are
 * empty); volumes = counts x sx sy sz; with S(M) = the voxels of M having a 6-neighbour outside M or outside the volume and
 * d_AB = for each voxel of S(A) the Euclidean distance in mm to the nearest voxel of S(B) (d_BA alike): hd_mm = max of both,
 * hd95_mm = np.percentile(hstack(d_AB, d_BA), 95) (linear interpolation), assd_mm = (mean d_AB + mean d_BA) / 2, all three
 * NaN when A or B is empty.  confusion_host (nullable) int64 [15][15]: [r][s] = voxels with reference class r and
 * segmentation class s.  Synchronises the stream.  SC_ERR_ARG for NULL pointers, bad dims, a spacing that is not finite
 * and > 0, or a label above 15 in either input (the message names it); outputs are untouched on an error. */
typedef struct { int64_t n_seg, n_ref, n_both;
                 double dice, vol_seg_mm3, vol_ref_mm3, hd_mm, hd95_mm, assd_mm; } sc_structure_metrics;  /* 72 bytes */
SC_API int sc_evaluate_segmentation(sc_ctx* ctx, const uint8_t* seg_dev, const uint8_t* ref_dev, const int32_t dims[3],
                                    const double spacing[3], sc_structure_metrics* metrics_host /* [14], class l at l-1 */,
                                    int64_t* confusion_host /* [15][15] or NULL */, void* stream);

/* ---- atlas registration ---------------------------------------------------------------
 * replaces: register_masks (base.py:483-551), i.e. niftyreg reg_aladin + reg_f3d + reg_resample, which map the template
 * T1 and its 15 structure priors onto the subject.  Not bit-compatible with niftyreg; its structure and conventions:
 *   - reference = the subject T1 (float32 [X][Y][Z]; its mask is the voxels != 0), floating = the template T1;
 *   - *_vox2mm: row-major 4x4 voxel -> mm matrices (what cnn_cort/nifti.py returns as .affine);
 *   - phi(x) = A [x; 1] + u(v) maps subject mm to template mm: A is the 3x4 top of `affine` (row-major 4x4, last row
 *     0 0 0 1); u is a cubic B-spline displacement in template mm whose control point (i, j, k) sits at subject voxel
 *     ((i-1) s, (j-1) s, (k-1) s), s = 5 voxels; grid [gx][gy][gz][3] float32 with g = floor((d - 1) / 5) + 4
 *     (sc_ffd_grid_dims).  Because the control points hold template mm, d F(phi(x)) / d c_k = beta_k(x) grad F(phi(x));
 *   - trilinear sampling in fp32 (in software); a point is inside the template when its voxel coordinate lies in [0, d-1]
 *     on every axis; outside, warped values are 0 and the subject voxel does not count towards the similarity;
 *   - NMI = (H_R + H_F) / H_RF, 64 bins, cubic B-spline Parzen windows on both axes; intensities mapped linearly to
 *     [2, 61] from [min, max] over the subject's mask and over every template voxel;
 *   - BE = mean over the interior control points of the squared second derivatives of u with respect to the grid
 *     coordinates (cross terms doubled), analytic at the control points; the FFD maximises J = (1 - 0.001) NMI - 0.001 BE.
 * sc_register_affine: A from the translation between the intensity centres of mass, then conjugate-gradient ascent of NMI
 * on a 4-level pyramid (factors 8, 4, 2, 1; levels where either image would have a dim below 16 are skipped).
 * sc_register_ffd: grid_dev (written) from a zero grid on a 3-level pyramid (factors 4, 2, 1; control points every 5
 * voxels of each level, refined exactly by B-spline subdivision between levels) for the given affine.
 * Deterministic: the same inputs give byte-identical results on every run.  Both synchronise the stream.
 * SC_ERR_ARG: NULL pointers, a dim below 8, a singular or non-finite matrix, an empty reference mask or no overlap of the
 * mask with the template (the message names the input). */
SC_API int sc_ffd_grid_dims(const int32_t ref_dims[3], int32_t grid_dims_out[3]);
SC_API int sc_register_affine(sc_ctx* ctx, const float* ref_dev, const int32_t ref_dims[3], const double ref_vox2mm[16],
                              const float* flo_dev, const int32_t flo_dims[3], const double flo_vox2mm[16], double affine_out[16],
                              void* stream);
SC_API int sc_register_ffd(sc_ctx* ctx, const float* ref_dev, const int32_t ref_dims[3], const double ref_vox2mm[16],
                           const float* flo_dev, const int32_t flo_dims[3], const double flo_vox2mm[16], const double affine[16],
                           float* grid_dev, void* stream);
/* replaces: reg_resample.  out_dev [X][Y][Z][channels] on the subject grid (ref_dims / ref_vox2mm) = the floating volume
 * [fX][fY][fZ][channels] (channels 1 or 15, channels-last) sampled trilinearly at phi(x), 0 outside; grid_dev NULL = affine only. */
SC_API int sc_warp_volume(sc_ctx* ctx, const float* flo_dev, const int32_t flo_dims[3], int channels, const double flo_vox2mm[16],
                          const double affine[16], const float* grid_dev, const int32_t ref_dims[3], const double ref_vox2mm[16],
                          float* out_dev, void* stream);
/* the objective at full resolution for a fixed (affine, grid) (parity tests of the kernels, as sc_dense_layer is for the
 * GEMMs): value_out = {NMI, BE, J} (BE = 0 and J = NMI when grid_dev is NULL); affine_grad_host[12] (nullable) = d NMI / d A
 * for the 12 entries of the 3x4 top of `affine`, row-major; grid_grad_dev (nullable, needs grid_dev) = d J / d grid. */
SC_API int sc_register_objective(sc_ctx* ctx, const float* ref_dev, const int32_t ref_dims[3], const double ref_vox2mm[16],
                                 const float* flo_dev, const int32_t flo_dims[3], const double flo_vox2mm[16], const double affine[16],
                                 const float* grid_dev, double value_out[3], double* affine_grad_host, float* grid_grad_dev,
                                 void* stream);
/* the registered sub-cortical mask (base.py:540-551, quirk Q11): (sum of channels 0..12 of the warped priors [X][Y][Z][15]) > 0,
 * dilated `iterations` times (sc_dilate_mask), as float32 0 / 1 [X][Y][Z]. */
SC_API int sc_prior_mask(sc_ctx* ctx, const float* priors_dev, const int32_t dims[3], int iterations, float* mask_dev, void* stream);

/* ---- resampling to the network's grid ------------------------------------------------
 * The network is defined in voxels (32-voxel patches, 3x3 taps) and its weights were trained on 1 mm isotropic images; with
 * [model] resample_mm the dense path runs on an isotropic grid of that voxel size and maps its output back to the scan's grid.
 * Per axis independently: the native grid has n voxels, the target grid m (cnn_cort/base.py:resample_dims), r = n / m; the
 * target grid keeps the native array axes and covers the same field of view (affine: native . [[diag(r), (r - 1) / 2], [0, 1]]).
 *   sc_resample_volume: native -> target.  Target index j sits at native coordinate x_j = (j + 0.5) r - 0.5; with h = max(r, 1)
 *     and w_ij = max(0, 1 - |i - x_j| / h) for 0 <= i < n, out_j = sum_i w_ij v_i / sum_i w_ij; the 3-D result is the separable
 *     product of the three 1-D filters.  r > 1: antialiasing triangle filter; r < 1: linear interpolation with the edge value
 *     held; r = 1: the identity, bit for bit.  Equal to torch's interpolate(mode='bilinear', antialias=True, align_corners=False)
 *     per pair of axes.  in_dev [X][Y][Z][channels] and out_dev [m0][m1][m2][channels] float32, channels-last, channels 1 or 15,
 *     filtered per channel.  The weights are convex: priors stay in [0, 1] and their per-voxel sum is kept.
 *   sc_map_proba_back: target -> native.  Native voxel v sits at target y = (v + 0.5) / r - 0.5 per axis, clamped to [0, m - 1];
 *     of its 8 trilinear neighbours those with non-zero weight and cand_dev != 0 are kept and their weights renormalised; the
 *     native probability vector is the weighted mean of their proba_dev rows [m0*m1*m2][15], the label its first arg-max.  A
 *     native voxel is written (label_dev uint8 [X][Y][Z], proba_out_dev float32 [X][Y][Z][15] when not NULL) only if it has at
 *     least one such neighbour and native_mask_dev (uint8 [X][Y][Z], NULL = every voxel) is non-zero there; every other voxel
 *     keeps what the outputs held.
 * Both accumulate in fp32 in a fixed order without atomics (the same inputs give byte-identical outputs); intermediates and the
 * per-axis weight tables live in the context.  SC_ERR_ARG, outputs untouched, for NULL required pointers, a dim below 1,
 * channels not 1 or 15 and an output that is its input; the message names the argument. */
SC_API int sc_resample_volume(sc_ctx* ctx, const float* in_dev, const int32_t in_dims[3], int channels, const int32_t out_dims[3],
                              float* out_dev, void* stream);
SC_API int sc_map_proba_back(sc_ctx* ctx, const float* proba_dev, const uint8_t* cand_dev, const int32_t target_dims[3],
                             const uint8_t* native_mask_dev, const int32_t native_dims[3], uint8_t* label_dev, float* proba_out_dev,
                             void* stream);

/* ---- scatter -------------------------------------------------------------------------
 * replaces: image[x,y,z] = y_pred and image_proba[x,y,z,c] = proba[:,c] (base.py:430-440) */
SC_API int sc_scatter(sc_ctx* ctx, const int32_t* xyz_dev, int64_t n, const int32_t* label_dev,
               const float* proba_dev, const int32_t dims[3], uint8_t* label_vol_dev,
               float* proba_vol_dev, void* stream);

/* ---- training ------------------------------------------------------------------------
 * replaces: one minibatch of nolearn's train_fn inside net.fit (nets.py:233-246):
 * training-mode forward (BN batch statistics, dropout p=.5), categorical cross-entropy,
 * backward.  Gradients land in the context's flat gradient buffer (parameter layout); the
 * slots of the BN running statistics receive this batch's mean / inv_std (applied by
 * sc_adam_step).  drop_masks_dev: NULL to draw masks from `seed`, or [n][3*540 + 540 + 540]
 * uint8 keep-masks per sample (axial|coronal|saggital l1drop in (c,h,w) order, f1_drop, f2_drop).
 * loss_dev: 1 float (sum of -log p over the batch divided by `n_global`). */
SC_API int sc_train_forward_backward(sc_ctx* ctx, const float* in1_dev, const float* in2_dev,
                              const float* in3_dev, const float* in4_dev, const uint8_t* y_dev,
                              int64_t n, int64_t n_global, uint64_t seed,
                              const uint8_t* drop_masks_dev, float* loss_dev, void* stream);
/* device pointers to the flat gradient / parameter buffers (SC_PARAM_FLOATS floats) so the
 * caller can all-reduce gradients in place (NCCL via torch.distributed). */
SC_API int sc_grad_buffer(sc_ctx* ctx, float** grads_dev);
SC_API int sc_param_buffer(sc_ctx* ctx, float** params_dev);
/* replaces: lasagne.updates.adam (nets.py:236-237): a_t = lr*sqrt(1-b2^t)/(1-b1^t);
 * p -= a_t * m / (sqrt(v) + eps) over the trainable entries, gradient multiplied by grad_scale first.
 * The slots of the BN running statistics in the gradient buffer carry the batch mean / inv_std
 * (summed over ranks by the all-reduce): s <- 0.9 s + 0.1 * slot * stat_scale (stat_scale = 1/world).
 * Marks the inference layouts stale; they are re-derived lazily by the next inference call. */
SC_API int sc_adam_step(sc_ctx* ctx, float lr, float beta1, float beta2, float eps, float grad_scale, float stat_scale, void* stream);
SC_API int sc_reset_optimizer(sc_ctx* ctx);
/* Data-parallel step as ONE kernel over NVLink peer memory: sum-all-reduce of the gradient buffers fused with sc_adam_step
 * (each rank reduces and updates its 1/world slice out of the peers' buffers and stores the new parameters into every peer;
 * csrc/fused_adam.cu).  One process per GPU: sc_fused_export writes 3 CUDA IPC handles (192 bytes: gradients, parameters,
 * flag page); the caller gathers the handles of all ranks (torch.distributed all_gather) and passes the world x 192 bytes,
 * in rank order, to sc_fused_attach on every rank (world <= 8).  sc_allreduce_adam_step must then be called by every rank
 * once per step, after sc_train_forward_backward on the same stream; it replaces all_reduce + sc_adam_step (the statistics
 * slots are averaged over the ranks).  All ranks end every step with bit-identical parameters. */
#define SC_IPC_BYTES 192
SC_API int sc_fused_export(sc_ctx* ctx, unsigned char* handles_out);
SC_API int sc_fused_attach(sc_ctx* ctx, int rank, int world, const unsigned char* all_handles);
SC_API int sc_allreduce_adam_step(sc_ctx* ctx, float lr, float beta1, float beta2, float eps, void* stream);
/* Synchronised BatchNorm for data-parallel training (SURVEY.md 5.8): the reference normalises over the whole batch of its
 * single device; with the hook set, the per-channel BatchNorm sums of the forward pass ({sum x, sum x^2}) and of the backward
 * pass ({sum dy, sum dy*xhat}) plus the element count are handed to `fn` as one small float64 device buffer right after they
 * are reduced locally; `fn` must sum it over all ranks IN PLACE, ordered on `stream` (an all-reduce of torch.distributed /
 * NCCL).  N ranks then reproduce the single-device step on the same global batch.  fn == NULL (default): per-GPU statistics.
 * With a hook the step is launched kernel by kernel (no CUDA graph). */
typedef int (*sc_allreduce_fn)(void* user, void* buf_dev /* double[count] */, int64_t count, void* stream);
SC_API int sc_set_allreduce_hook(sc_ctx* ctx, sc_allreduce_fn fn, void* user);
/* evaluation pass of nolearn's eval_fn: mean CE loss and accuracy numerators over a batch
 * in deterministic mode; out2_dev = {sum of -log p[y], number of correct argmax}. */
SC_API int sc_eval_batch(sc_ctx* ctx, const float* in1_dev, const float* in2_dev, const float* in3_dev,
                  const float* in4_dev, const uint8_t* y_dev, int64_t n, float* out2_dev, void* stream);

/* ---- fine-tuning on a new domain: frozen trunk, cached trunk features, head-only steps ------------------------------
 * Supervised domain adaptation as in Kushibar et al. (Sci. Rep. 2019): keep the convolutional layers, retrain the fully
 * connected part on a few labelled target-domain samples.
 *   trunk = every <view>_ch_conv1..5 (W), <view>_ch_conv1..5_bn (beta, gamma, mean, inv_std) and <view>_ch_prelu1..5 array of
 *           the three views; head = every other array (d1 x3, FC1, fc_2, out_layer and their PReLUs).
 * The trunk is evaluated in deterministic mode, with the STORED BatchNorm statistics: a sample's features then do not depend
 * on its minibatch (so they are computed once and cached), and the batch statistics of a single target image cannot shift the
 * frozen layers.  This deliberately differs from a training-mode forward pass with frozen weights.  The head trains with the
 * semantics of sc_train_forward_backward: dropout p = .5 at *_l1drop (on the cached features), f1_drop and f2_drop with the same
 * [n][2700] mask layout and the same hash3(seed, i) masks, softmax cross-entropy divided by n_global, Lasagne Adam.
 * Feature rows (public layout): float32 [N][3][540]; per view, entry k = c*9 + h*3 + w is the flattened conv5 activation after
 * BatchNorm and PReLU, i.e. the input of <view>_d1 before dropout.
 * All four calls return SC_ERR_ARG with the SIMT back-end selected ("gemm" = 0; sc_freeze_trunk(ctx, 0) excepted), for NULL
 * required pointers and for bad sizes; the message names the argument. */
/* trunk of the three views on [n][1][32][32] patches (the tensor-core patchwise trunk of sc_forward) -> feats_dev [n][3][540]. */
SC_API int sc_trunk_features(sc_ctx* ctx, const float* in1_dev, const float* in2_dev, const float* in3_dev, int64_t n,
                             float* feats_dev, void* stream);
/* One training step of the head on rows r = idx_dev[i] (r = i when idx_dev is NULL), i < n <= 16384, of a feature table
 * feats_dev [N][3][540] with the atlas rows atlas_rows_dev [N][15] and labels labels_dev [N] (uint8 0..14) that a training set
 * holds on the device.  n_global, seed, drop_masks_dev and loss_dev as for sc_train_forward_backward (the masks are per batch
 * entry i).  Gradients land in the context's gradient buffer; every trunk entry of it, the BatchNorm-statistics slots included,
 * is exactly 0 afterwards.  Indices are device data and are not range-checked (0 <= idx[i] < N is the caller's to guarantee).
 * Captured as a CUDA graph per (n, n_global, injected masks, tables, idx NULL or not) like the full step ("train_graph"). */
SC_API int sc_head_train_forward_backward(sc_ctx* ctx, const float* feats_dev, const float* atlas_rows_dev, const uint8_t* labels_dev,
                                          const int64_t* idx_dev, int64_t n, int64_t n_global, uint64_t seed,
                                          const uint8_t* drop_masks_dev, float* loss_dev, void* stream);
/* deterministic head on the same rows (the validation pass of fine-tuning): out2_dev = {sum of -log p[y], number of correct
 * arg-max}, as sc_eval_batch reports for the patches the features came from. */
SC_API int sc_head_eval_batch(sc_ctx* ctx, const float* feats_dev, const float* atlas_rows_dev, const uint8_t* labels_dev,
                              const int64_t* idx_dev, int64_t n, float* out2_dev, void* stream);
/* frozen != 0: sc_adam_step and sc_allreduce_adam_step leave every trunk entry untouched (parameter, Adam moments, BatchNorm
 * running statistics), and sc_train_forward_backward returns SC_ERR_STATE; 0 restores the default.  Inference is unaffected.
 * Synchronises the device. */
SC_API int sc_freeze_trunk(sc_ctx* ctx, int frozen);

#ifdef __cplusplus
}
#endif
#endif /* SUBCORT_B200_H */
