// Shared declarations of the subcort_b200 library (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>
#include <utility>
#include <vector>

#include "../../include/subcort_b200.h"

namespace sc {

void set_error(const char* fmt, ...);

#define SC_CUDA(expr)                                                                        \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      sc::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));   \
      return SC_ERR_CUDA;                                                                    \
    }                                                                                        \
  } while (0)

#define SC_CHECK(cond, code, ...)   \
  do {                              \
    if (!(cond)) {                  \
      sc::set_error(__VA_ARGS__);   \
      return code;                  \
    }                               \
  } while (0)

#define SC_TRY(expr)           \
  do {                         \
    int _s = (expr);           \
    if (_s != SC_OK) return _s;\
  } while (0)

// ---------------------------------------------------------------------------------------
// Parameter table: offsets (in floats) into the flat pickle-ordered blob
// (nets/<name>/<name>.pkl, SURVEY.md 2.4; graph order of cnn_cort/nets.py:170-231).
// ---------------------------------------------------------------------------------------
constexpr int kConvCin[5] = {1, 20, 20, 40, 40};
constexpr int kConvCout[5] = {20, 20, 40, 40, 60};

struct BranchOff {
  int convW[5];   // (Cout, Cin, 3, 3)
  int bn[5][4];   // beta, gamma, mean, inv_std
  int alpha[5];   // PReLU
  int d1W, d1b, d1alpha;  // (540,180), (180), (180)
};
struct ParamOff {
  BranchOff br[3];
  int fc1W, fc1b, a1;   // (540,540) (540) (540)
  int fc2W, fc2b, a2;   // (555,270) (270) (270)
  int outW, outb;       // (270,15) (15)
  int total;
};
inline ParamOff make_param_off() {
  ParamOff P;
  int o = 0;
  for (int b = 0; b < 3; ++b) {
    for (int l = 0; l < 5; ++l) {
      P.br[b].convW[l] = o; o += kConvCout[l] * kConvCin[l] * 9;
      for (int k = 0; k < 4; ++k) { P.br[b].bn[l][k] = o; o += kConvCout[l]; }
      P.br[b].alpha[l] = o; o += kConvCout[l];
    }
    P.br[b].d1W = o; o += 540 * 180;
    P.br[b].d1b = o; o += 180;
    P.br[b].d1alpha = o; o += 180;
  }
  P.fc1W = o; o += 540 * 540; P.fc1b = o; o += 540; P.a1 = o; o += 540;
  P.fc2W = o; o += 555 * 270; P.fc2b = o; o += 270; P.a2 = o; o += 270;
  P.outW = o; o += 270 * 15; P.outb = o; o += 15;
  P.total = o;
  return P;
}

// ---------------------------------------------------------------------------------------
// Derived inference layouts (device)
// ---------------------------------------------------------------------------------------
// GEMM operand geometry: every K is padded to 576 = 9 blocks of 64.  Activation rows are 576 floats
// wide in both modes: plain fp32 (SIMT back-end), or -- for the tcgen05 back-end -- per 64-wide block
// 64 bf16 "hi" values followed by 64 bf16 "lo" values (x = hi + lo to ~2^-17): the split-precision
// operands of the three-MMA bf16x3 product (xh*wh + xh*wl + xl*wh), same bytes as fp32.
constexpr int kFeat = 540;       // concat of the three d1 outputs
constexpr int kFeatLd = 576;     // row stride of the feature buffer (K of FC1)
constexpr int kH1 = 555;         // FC1 out (540) + atlas (15)
constexpr int kH1Ld = 576;       // row stride (K of fc_2)
constexpr int kH2 = 270;
constexpr int kH2Ld = 272;
constexpr int kC5Ld = 64;        // conv5 output channels padded 60 -> 64 (NHWC)
constexpr int kD1K = 9 * kC5Ld;  // 576: K of d1 as a 3x3 dilation-4 conv over conv5 output

struct GemmW {      // one dense layer prepared for both GEMM back-ends
  float* w_kn;      // [Kpad][Npad] row-major fp32 (SIMT path), zero padded
  float* w_nk;      // [Npad][Kpad] K-major split bf16 hi|lo blocks (tcgen05 path), zero padded
  float* bias;      // [Npad]  (BN shift for the conv layers)
  float* alpha;     // [Npad] (PReLU; 1 where identity)
  float* scale;     // [Npad] multiplies the accumulator before the bias (BN scale), or nullptr = 1
  int K, N, Kpad, Npad;
  int k_used = 0;   // columns of the padded K row that can be non-zero (0 = all of Kpad): the tcgen05 GEMM skips the k-steps beyond
};

struct SweepW {     // one conv layer prepared for the strip-sweep tcgen05 kernel (conv_sweep.cu)
  float* panels;    // [npanels][6*bn][64] bf16: rows 0..3bn-1 = W hi stacked over the filter rows [W_ky2 | W_ky1 | W_ky0]
                    // (bn rows each), 3bn..6bn-1 = W lo stacked alike; column block (gk & 3) of panel gk >> 2 holds
                    // k-step gk = kx * ksteps + ci / 16 (flipped taps, zero padded)
  float* panels_pair;  // the same for the CTA-pair kernel: per panel the rows of rank 0 then rank 1, each W hi | W lo of its
                       // 1.5 bn stacked rows (rank 0: [W_ky2 | W_ky1[0, bn/2)], rank 1: [W_ky1[bn/2, bn) | W_ky0])
  float* scale;     // BN folded scale / shift and PReLU slope, padded to 64 with zeros
  float* shift;
  float* alpha;
  int bn, ksteps, npanels;   // npanels = ceil(3 * ksteps / 4)
};

// bf16 element offsets of the hi part of weight (output channel o, filter row ky, column kx, input channel k) in the
// plain and pair panels of SweepW; the lo parts lie 3 bn (plain) and 1.5 bn (pair) rows further
__host__ __device__ inline void sweep_panel_pos(int o, int ky, int kx, int k, int ksteps, int bn, size_t& plain, size_t& pair) {
  const int gk = kx * ksteps + (k >> 4), kk = (gk & 3) * 16 + (k & 15), panel = gk >> 2;
  const int sr = (2 - ky) * bn + o, hb = 3 * bn / 2;   // stacked row; stacked rows per CTA of a pair
  plain = ((size_t)panel * 6 * bn + sr) * 64 + kk;
  pair = ((size_t)(panel * 2 + sr / hb) * 3 * bn + sr % hb) * 64 + kk;
}

struct Conv1Consts { float w[9 * 20]; float scale[20], shift[20], alpha[20]; };   // conv1 taps + folded BN + PReLU, passed by value

struct BranchW {
  Conv1Consts c1_host;  // host copy of conv1's constants: kernel parameter (constant bank) of conv1_wide_kernel
  float* c1_w;          // [9][20]  flipped taps, tap = ky*3+kx
  float* conv_w[5];     // l=1..4 used: [Cin][9][Cout] flipped (conv2..conv5)
  float* scale[5];      // BN folded: gamma*inv_std
  float* shift[5];      // beta - mean*scale
  float* alpha[5];
  SweepW conv_sw[5];    // l=1..4: conv2..conv5 for the strip-sweep kernel
  GemmW d1;             // patchwise: K=540 (c*9+h*3+w order)
  GemmW d1_dense;       // dense: K=576 (tap*64+ci), same N
};

struct Workspace {
  void* ptr = nullptr;
  size_t bytes = 0;
};

// per-kernel-class timing with CUDA events on the launching stream (sc_set_option "profile")
enum ProfClass {
  PC_GATHER = 0, PC_NONZERO, PC_SCATTER, PC_PATCH_BRANCH, PC_CONV1, PC_CONV2, PC_CONV3, PC_CONV4, PC_CONV5,
  PC_GEMM_D1, PC_GEMM_FC1, PC_GEMM_FC2, PC_ATLAS, PC_OUT, PC_POOL, PC_TRAIN_FWD, PC_TRAIN_BWD, PC_ADAM, PC_EVALUATE, PC_REGISTER, PC_MC, PC_COUNT
};

// counter-based random bits (splitmix64 finaliser): the dropout keep masks of the training step and of Monte-Carlo dropout
__host__ __device__ inline uint32_t hash3(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (idx + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return (uint32_t)((z ^ (z >> 31)) >> 16);
}
// keep bits per dropout pass: [3][540] *_l1drop (k = c*9 + h*3 + w) | [540] f1_drop | [540] f2_drop
constexpr int kDropUnits = 2700;
struct ProfEvent { int cls; cudaEvent_t a, b; };

}  // namespace sc

struct sc_ctx {
  int device = 0;
  int sm_count = 0;
  bool weights_loaded = false;
  int gemm_backend = 1;          // 1 tcgen05 (the product path); 0 = exact-fp32 SIMT cross-check, tests only
  int64_t chunk_voxels = 1 << 20;
  int64_t launches = 0;
  sc::ParamOff off;
  float* params = nullptr;       // master copy, pickle order
  float* grads = nullptr;        // same layout
  float* adam_m = nullptr;
  float* adam_v = nullptr;
  uint8_t* trainable = nullptr;  // 1 where the entry is trainable
  int64_t adam_t = 0;
  float* derived = nullptr;      // arena for the derived layouts
  size_t derived_floats = 0;
  sc::BranchW br[3];
  sc::GemmW fc1, fc2;
  float* out_w = nullptr;        // [270][16] out_layer weights (fp32; SIMT kernel and the fused epilogue of fc_2)
  float* out_b = nullptr;        // [16]
  sc::Workspace ws;              // inference scratch (grow-only)
  sc::Workspace ws_train;        // staging of the host entry points, scan preparation, eval scratch
  sc::Workspace ws_fit;          // training step: staged inputs, saved activations, gradients of activations
  sc::Workspace ws_eval;         // sc_evaluate_segmentation: distance fields, envelope stacks and distance lists of one class box
  sc::Workspace ws_reg;          // registration: pyramids, histogram, adjoint passes, control-point grids
  double* h_reg = nullptr;       // pinned: the optimiser's per-trial read-backs
  int reg_iters[8] = {};         // accepted steps of the last registration per level: affine 0..3, FFD 4..6
  // training step as a CUDA graph (one per (batch, global batch, injected masks) shape): the three branches run on
  // three captured streams; rebuilt when the arena moves
  struct TrainGraph { int n; long long n_global; int injected; int backend; void* arena; cudaGraphExec_t exec; int launches; };
  std::vector<TrainGraph> train_graphs;
  cudaStream_t train_side[2] = {nullptr, nullptr};
  cudaEvent_t train_ev[8] = {};
  int train_graph_on = 1;        // sc_set_option("train_graph", 0): launch the step kernel by kernel (profiling, debugging)
  // fused all-reduce + Adam over peer memory (fused_adam.cu): peers' buffers opened through CUDA IPC
  unsigned* peer_flags = nullptr;
  float* peer_grads[8] = {}; float* peer_params[8] = {}; unsigned* peer_flagp[8] = {};
  int peer_rank = 0, peer_world = 0; unsigned peer_step = 0;
  sc_allreduce_fn ar_hook = nullptr;   // synchronised BatchNorm: sums the BN reduction buffers over the ranks (sc_set_allreduce_hook)
  void* ar_user = nullptr;
  void* train_panels = nullptr;  // sweep weight panels of the training step, re-derived on the device every step
  void* train_dense_w = nullptr; // dense weights of the training step in the two GEMM operand layouts, re-derived every step
  struct TrainDenseW { float* wnk; float* wkn; float* bias; };
  TrainDenseW train_dw[6];       // d1 x3, FC1, fc_2, out_layer
  sc::SweepW train_sw[3][5][2];  // [branch][layer 1..4][forward | dgrad]
  float* train_consts = nullptr; // 1024 ones | 1024 zeros (identity epilogue constants of the training kernels)
  int64_t* d_count = nullptr;    // device scalar for stream compaction
  int64_t* h_count = nullptr;    // pinned
  void* tc_state = nullptr;      // tcgen05 back-end state (tensor-map encoder entry point)
  int tc_timing_cls = -1;        // ProfClass whose persistent launches record per-role wait cycles (debug)
  unsigned long long* tc_timing_buf = nullptr;   // [sm_count][8], overwritten by every instrumented launch
  int train_wgrad_mn = 1;        // conv weight gradients from the pixel-major maps (MN-major operands) instead of planar transposed copies
  int train_fused_stats = 1;     // training forward: BatchNorm statistics accumulated in the sweep epilogues (off: a separate pass over the stored maps)
  int tc_skip = 1;               // dense path with a sparse candidate mask: the conv sweeps skip the items no candidate needs
  int tc_compact = 1;            // dense path with a candidate mask: the FC head runs on the compacted candidate rows only
  int32_t* h_slab_cnt = nullptr; // pinned: candidates per slab
  float* mc_w = nullptr;         // Monte-Carlo dropout: the row-masked split weights (w_nk) of d1 x3, FC1 and fc_2 for one pass
  unsigned char* tile_flags = nullptr;   // d1 with a row map: per-tile "has a candidate" flags (device, grow-only)
  size_t tile_flags_cap = 0;
  cudaEvent_t compact_ev = nullptr;
  int gather_ctas_per_sm = 0;    // > 0: persistent gather grid of that many CTAs per SM; 0 (default, measured fastest) = one CTA per 32-candidate group
  cudaStream_t copy_stream = nullptr;   // sc_segment_volume_host: the 1 GB atlas upload overlaps the conv phase
  cudaEvent_t copy_ev[2] = {nullptr, nullptr};
  cudaEvent_t atlas_ready = nullptr;    // when set, segment_volume waits for it before its first use of the atlas (phase 2)
  // chunked upload: atlas_chunk_ev[i] fires when the x-planes [0, (i + 1) * atlas_chunk_nx) of the atlas are on the device;
  // a slab of phase 2 only waits for the chunks that cover it (atlas_chunks > 0 replaces the single event above)
  cudaEvent_t atlas_chunk_ev[64] = {};
  int atlas_chunks = 0, atlas_chunk_nx = 0;
  // pageable host atlas: a helper thread issues the (then blocking) chunk copies; the consumer must not wait for an
  // event before the helper has recorded it: chunks recorded so far (nullptr = all recorded before the kernels were launched)
  std::atomic<int>* atlas_recorded = nullptr;
  bool profile = false;
  std::vector<sc::ProfEvent> prof_live;
  std::vector<sc::ProfEvent> prof_free;
  bool derived_dirty = false;    // master parameters changed since the inference layouts were derived
  // kernels whose MaxDynamicSharedMemorySize has been raised on THIS context's device (the attribute is per device)
  std::vector<std::pair<const void*, int>> smem_attr;
};

namespace sc {
int ensure_ws(Workspace& ws, size_t bytes);
// cudaFuncAttributeMaxDynamicSharedMemorySize applies per device: remembered per context, never in a process-wide static
int ensure_smem_attr(sc_ctx* ctx, const void* kernel, int bytes);

const char* prof_class_name(int cls);
// one scope per kernel launch: an NVTX range named after the kernel class (header-only NVTX v3: a no-op unless a
// profiler is attached) and, with sc_set_option("profile", 1), a pair of CUDA events on the launching stream
struct ProfScope {
  sc_ctx* ctx; cudaStream_t st; ProfEvent ev; bool on;
  ProfScope(sc_ctx* c, int cls, cudaStream_t s) : ctx(c), st(s), on(c->profile) {
    nvtxRangePushA(prof_class_name(cls));
    if (!on) return;
    if (!ctx->prof_free.empty()) { ev = ctx->prof_free.back(); ctx->prof_free.pop_back(); }
    else { cudaEventCreate(&ev.a); cudaEventCreate(&ev.b); }
    ev.cls = cls;
    cudaEventRecord(ev.a, st);
  }
  ~ProfScope() {
    if (on) {
      cudaEventRecord(ev.b, st);
      ctx->prof_live.push_back(ev);
    }
    nvtxRangePop();
  }
};

// gather.cu
// row m of a box slab <-> voxel (x0 + m / (by*bz), y0 + (m / bz) % by, z0 + m % bz) of a [X][Y][Z] volume
struct OutGeo { int x0, y0, z0, by, bz, Y, Z; };

int launch_gather(sc_ctx* ctx, const float* vol, const int32_t* dims, const float* atlas, int bg_fix,
                  const int32_t* xyz, int64_t n, float* ax, float* co, float* sa, float* atlas_out, cudaStream_t st);
// ordered compaction of the candidate rows of every slab of a box (slab = nx_per_slab x-planes): rowmap[dense row] = compact
// row or -1, rowvox[slab base + compact row] = dense row inside the slab, cnt[slab] = candidates; scratch: 2 ints per 2048 rows
int launch_slab_compact(sc_ctx* ctx, const uint8_t* cand, const OutGeo& box, int bx, int nx_per_slab, int32_t* rowmap, int32_t* rowvox,
                        int32_t* cnt, int32_t* scratch, cudaStream_t st);
int launch_center_labels(sc_ctx* ctx, const uint8_t* lab, const int32_t* dims, const int32_t* xyz, int64_t n,
                         uint8_t* y, cudaStream_t st);
int launch_gather_samples(sc_ctx* ctx, const sc_scan* scans, int n_scans, const int32_t* samples, const float* atlas_rows,
                          const uint8_t* labels, const int64_t* idx, int64_t n, float* ax, float* co, float* sa,
                          float* atlas_out, uint8_t* y_out, cudaStream_t st);
int launch_nonzero(sc_ctx* ctx, const void* vol, int elem_bytes, const int32_t* dims, int32_t* xyz,
                   int64_t capacity, int64_t* n_out_host, cudaStream_t st);
int launch_dilate(sc_ctx* ctx, const uint8_t* mask, const int32_t* dims, int iterations, uint8_t* out, cudaStream_t st);
int launch_scatter(sc_ctx* ctx, const int32_t* xyz, int64_t n, const int32_t* label, const float* proba,
                   const int32_t* dims, uint8_t* label_vol, float* proba_vol, cudaStream_t st);

// prep.cu : scan preparation on the device (array-order import, normalisation, candidate mask, bounding box)
int import_volume(sc_ctx* ctx, const void* src, int elem_bytes, const int32_t* dims, int channels, void* dst, cudaStream_t st);
int upload_volume_box(sc_ctx* ctx, const void* src_host, int elem_bytes, const int32_t* dims, int channels, int fortran_order,
                      const int32_t* box, void* staging_dev, void* dst, cudaStream_t st);
int normalise_volume(sc_ctx* ctx, const void* vol, int dtype, const int32_t* dims, float* out, double* mean_std_host, cudaStream_t st);
int candidate_mask(sc_ctx* ctx, const void* vol, int dtype, const int32_t* dims, uint8_t* mask, cudaStream_t st);
int mask_bbox(sc_ctx* ctx, const uint8_t* mask, const int32_t* dims, int32_t* box_host, int64_t* count_host, cudaStream_t st);

// postproc.cu : connected-component post-processing of a label volume
int post_process(sc_ctx* ctx, const uint8_t* seg, const uint8_t* mask, const int32_t* dims, uint8_t* out, cudaStream_t st);

// evaluate.cu : per-structure Dice, volumes and surface distances of a label volume against a reference
int evaluate_segmentation(sc_ctx* ctx, const uint8_t* seg, const uint8_t* ref, const int32_t* dims, const double* spacing,
                          sc_structure_metrics* metrics, int64_t* confusion, cudaStream_t st);

// register.cu : affine + B-spline FFD registration of the template to the subject (NMI), warps and the prior mask
void ffd_grid_dims(const int32_t* ref_dims, int32_t* grid_dims);
int register_affine(sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                    const double* fv, double* affine_out, cudaStream_t st);
int register_ffd(sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                 const double* fv, const double* affine, float* grid_out, cudaStream_t st);
int register_objective(sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                       const double* fv, const double* affine, const float* grid, double* value, double* agrad, float* ggrad,
                       cudaStream_t st);
int warp_volume(sc_ctx* ctx, const float* flo, const int32_t* fdims, int channels, const double* fv, const double* affine, const float* grid,
                const int32_t* rdims, const double* rv, float* out, cudaStream_t st);
int prior_mask(sc_ctx* ctx, const float* priors, const int32_t* dims, int iterations, float* out, cudaStream_t st);

// weights.cu
int derive_weights(sc_ctx* ctx, cudaStream_t st);

// gemm_simt.cu : C = prelu(A*W + b), implicit-GEMM with taps
struct GemmProblem {
  const float* A;       // A(m, y, z, tap, k) = A[z*a_zs + y*a_ys + m*lda + tap_off[tap] + k]
  int64_t lda, a_ys, a_zs;
  int ntaps;            // 1 (dense layer) or 9 (3x3 conv)
  int64_t tap_off[9];
  int kc;               // K per tap (multiple of 4)
  float* C;             // C(m, y, z, n) = C[z*c_zs + y*c_ys + m*ldc + n]
  int64_t ldc, c_ys, c_zs;
  int M, Y, Z;          // rows per (y,z) line, lines, planes
  // tcgen05 back-end: the same A described for a 4-D TMA tensor map (k, pixel, line, plane)
  const float* a_base;  // start of the whole buffer (16 B aligned)
  int64_t a_dims[4];    // extents: k, pixels per line, lines, planes
  int64_t a_strides[3]; // element strides of pixel, line, plane
  int tap_dx[9], tap_dy[9];  // tap shifts in pixels / lines
  int tap_dz[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // ... / planes (tcgen05 back-end only)
  int a_y0, a_z0;       // line / plane offset of this launch inside the buffer
  int prof_cls;         // ProfClass of this launch
  int k_used;           // conv layers: real input channels per tap (the rest of the 64-wide block is zero); 0 = all
  int n_store;          // columns written (<= w.Npad)
  int c_col0;           // first output column inside the C row (C points at the row start)
  int out_split;        // write C rows in the split bf16 hi|lo block layout (they feed a tcgen05 GEMM)
  // candidate compaction (tcgen05 pair kernel): d1 writes row r of its dense slab to C row rowmap[r] (skipped when < 0);
  // FC1 finds the voxel of its compact row m through rowvox[m] (atlas lookup)
  const int32_t* rowmap = nullptr;
  const int32_t* rowvox = nullptr;
  const float* atlas = nullptr;            // tcgen05 pair kernel (FC1): write the atlas prior of every row (with the background
  OutGeo ageo;                             // fix of base.py:392-394) into columns 540..554 and zeros up to 575
  const struct SoftmaxOut* sm = nullptr;   // tcgen05 back-end, fc_2 only: out_layer + softmax / argmax in the epilogue instead of the row store
  int a_swap = 0;       // tensor-map dimension order is (k, pixel, plane, line) instead of (k, pixel, line, plane)
  // with sm: Monte-Carlo dropout pass instead of the store -- row m adds {softmax p[0..14], sum_c p_c ln p_c} to
  // mc_acc[m * 16 ..] (mc_first: stores instead of adding)
  float* mc_acc = nullptr;
  int mc_first = 0;
};
int launch_gemm(sc_ctx* ctx, const GemmProblem& p, const GemmW& w, cudaStream_t st);
// plain [M][lda] row-major A, one tap: fills both the pointer form and the tensor-map form
inline void gemm_problem_rows(GemmProblem& p, const float* A, int64_t lda, int kc, int M) {
  p.c_col0 = 0; p.out_split = 0; p.k_used = 0; p.a_swap = 0;
  p.A = A; p.lda = lda; p.a_ys = p.a_zs = 0; p.ntaps = 1; p.tap_off[0] = 0; p.kc = kc;
  p.M = M; p.Y = p.Z = 1; p.c_ys = p.c_zs = 0;
  p.a_base = A; p.a_dims[0] = kc; p.a_dims[1] = M; p.a_dims[2] = p.a_dims[3] = 1;
  p.a_strides[0] = lda; p.a_strides[1] = p.a_strides[2] = (int64_t)M * lda;
  for (int t = 0; t < 9; ++t) p.tap_dx[t] = p.tap_dy[t] = 0;
  p.a_y0 = p.a_z0 = 0;
}
// rows of h2 -> softmax / argmax.  geo == nullptr: row m writes proba[m], label32[m].
// geo != nullptr: row m is voxel (ix,iy,iz) of a box slab; results go to the volume-shaped
// outputs (label8 / proba) at that voxel, skipped where mask[voxel] == 0.
// out_layer + softmax fused into the epilogue of the tcgen05 fc_2 GEMM: where the results of row m go
struct SoftmaxOut { float* proba; int32_t* label32; uint8_t* label8; const uint8_t* mask; OutGeo geo; int use_geo;
                    const int32_t* rowvox; };   // rowvox != nullptr: GEMM row m is the compacted candidate whose slab row is rowvox[m]
int launch_out_softmax(sc_ctx* ctx, const float* h2, int64_t n, float* proba, int32_t* label32, uint8_t* label8,
                       const uint8_t* mask, const OutGeo* geo, cudaStream_t st);

// gemm_tc.cu : tcgen05 / TMEM / TMA back-end for the same problem
int tc_init(sc_ctx* ctx);
void tc_destroy(sc_ctx* ctx);
int launch_gemm_tc(sc_ctx* ctx, const GemmProblem& p, const GemmW& w, cudaStream_t st);
int launch_split_rows(sc_ctx* ctx, const float* in, int64_t rows, float* out, cudaStream_t st);  // [rows][576] plain -> split

// one view of a box of the volume (or a stack of patches) as slices x rows x cols
struct ViewGeo {
  int64_t ss, rs, cs;   // element strides of slice / row / col in the [X][Y][Z] volume
  int s0, ns;           // slice range of the box along the view's slice axis
  int r0, c0;           // box origin inside the slice
  int br, bc;           // box extent (rows, cols)
  int R, C;             // full slice extent (zero outside)
};

// conv_sweep.cu : conv1 (1 -> 20 channels) straight from the volume / patches into a wide-row F32CH map
int launch_conv1_wide(sc_ctx* ctx, const float* vol, const ViewGeo& g, int ns, const Conv1Consts& cw, float* out, int outR, int outC,
                      cudaStream_t st);
// conv_sweep.cu : strip-sweep 3x3 dilated conv (+ fused stride-1 max-pool) over wide-row maps.
// in_fmt / out_fmt: 1 = 128 B pixels (32 bf16 hi | 32 lo), 0 = 256 B pixels (64 hi | 64 lo)
// Sparse candidate masks: an output position (row r, slice s, col c) of a layer is needed only if a candidate voxel (i, j) of slice s
// has r - reach <= i <= r and c - reach <= j <= c (reach = rows_out - br: the receptive-field extent downstream of the layer).
// occ[i * ns + s]: bit jb set when row i of slice s holds a candidate in columns [32 jb, 32 jb + 32) (launch_view_occupancy);
// the sweep then skips the items (strip x row segment) no candidate needs.  flags: scratch of >= the number of items bytes.
// training forward: per-channel sum / sum of squares of the raw conv output over the valid H x H region of every patch, accumulated
// into sums[c][2] (doubles) by the sweep's epilogue -- the BatchNorm statistics without a separate pass over the map
struct SweepStats { double* sums; int H, pitch; };
struct SweepSkip { const uint32_t* occ; int br, bc, ns, C1; uint8_t* flags; };
int launch_view_occupancy(sc_ctx* ctx, const uint8_t* cand, const ViewGeo& g, uint32_t* occ, cudaStream_t st);
int launch_conv_sweep(sc_ctx* ctx, const SweepW& w, int layer, const float* in, int in_fmt, float* out, int out_fmt,
                      int Pw, int R, int rows_out, int dil, int pool, int prof_cls, cudaStream_t st, int in_dx = 0, int in_dy = 0,
                      const SweepSkip* skip = nullptr, const struct SweepStats* stats = nullptr);

// patch_forward.cu
int launch_branch_patches(sc_ctx* ctx, int branch, const float* patches, int64_t n, float* c5_out /*[n][540]*/,
                          cudaStream_t st);
int forward_patches(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, const float* in4, int64_t n,
                    float* proba, int32_t* label, cudaStream_t st);

// dense.cu
struct ConvArgs {
  const float* in; int inR, inLd;       // planar [ns][CIN][inR][inLd] (raw, before the folded pool)
  float* out; int outR, outC, outLd;    // planar [ns][COUT][outR][outLd] or NHWC [ns][outR][outC][64]
  const float* w;                       // [CIN][9][COUT]
  const float* scale; const float* shift; const float* alpha;
  int ns; int round_out;                // round_out: write the NHWC map in the split bf16 hi|lo layout
};
int launch_conv3x3(sc_ctx* ctx, int cin, int cout, const ConvArgs& a, int prof_cls, cudaStream_t st);
int launch_conv1_patches(sc_ctx* ctx, const float* patches, int n, const float* w, const float* scale, const float* shift,
                         const float* alpha, float* out, cudaStream_t st);
size_t branch_patches_tc_bytes(int64_t n);
int branch_patches_tc(sc_ctx* ctx, int branch, const float* patches, int64_t n, float* scratch, float* feats /*[n][576] split*/,
                      cudaStream_t st);
// Monte-Carlo dropout over the FC head (mc_dropout.cu): `samples` passes with the keep masks hash3(seed, t * 2700 + j)
struct McArgs { int samples; uint64_t seed; float* entropy; float* mi; };
int segment_volume(sc_ctx* ctx, const float* vol, const int32_t* dims, const float* atlas, const int32_t* box,
                   const uint8_t* cand, uint8_t* label_vol, float* proba_vol, cudaStream_t st, const McArgs* mc = nullptr);

// mc_dropout.cu : the masked weights of one pass and the per-voxel statistics of a slab
struct McWeights { GemmW d1[3], fc1, fc2; };
int mc_prepare(sc_ctx* ctx, McWeights& w);
int launch_mc_mask(sc_ctx* ctx, uint64_t seed, int t, cudaStream_t st);
int launch_mc_finalize(sc_ctx* ctx, const float* acc, int64_t rows, int samples, const int32_t* rowvox, const OutGeo& geo,
                       const uint8_t* mask, uint8_t* label, float* proba, float* entropy, float* mi, cudaStream_t st);

// train_tc.cu : the convolutional part of the training step on the tensor cores (split-bf16 wide-row maps)
constexpr float kBnEps = 1e-4f;
struct TcBranchBuf {
  float* X[5]; float* A[5]; uint16_t* AT[5]; uint8_t* idx[5]; float* mean[5]; float* istd[5];
  float* frame; float* dA; uint16_t* DT; float* dX0; double* sums;
};
size_t tc_branch_bytes(int n);
int tc_carve_branch(TcBranchBuf& T, char* base, int n);
int tc_branch_forward(sc_ctx* ctx, int b, const TcBranchBuf& T, const float* patches, const float* wf0, int n, const uint8_t* masks,
                      float* F5, cudaStream_t s);
int tc_branch_backward(sc_ctx* ctx, int b, const TcBranchBuf& T, const float* patches, const float* dF5, int dF5_ld, const uint8_t* masks, int n,
                       cudaStream_t s);
// train_dense.cu : the dense layers of the training step as split-bf16 tcgen05 GEMMs
constexpr int kTrainZeros = 1024;   // ctx->train_consts: 1024 ones | 1024 zeros (identity epilogue constants)
struct TcDenseBuf {
  int npad;                                  // batch rounded up to 64: K of the wgrad GEMMs
  char* zero_begin; size_t zero_bytes;       // split operands whose padding must read as zero: cleared every step
  float *F5s[3], *F5T[3], *Z1[3], *dZ1s[3], *dZ1T[3], *dF5[3], *gW1[3];
  float *CATs, *CATT, *ZF1, *CAT2s, *CAT2T, *ZF2, *H2s, *H2T, *ZO, *dZOs, *dZOT, *dH2, *dZF2s, *dZF2T, *dCAT2, *dZF1s, *dZF1T, *dCAT;
  float *gWfc1, *gWfc2, *gWout;
};
int tc_train_prepare(sc_ctx* ctx);      // persistent buffers: allocated outside any stream capture
int tdense_prepare(sc_ctx* ctx);
size_t tdense_bytes(int n);
void tdense_carve(TcDenseBuf& D, char* base, int n);
int tdense_branch_forward(sc_ctx* ctx, int b, const TcDenseBuf& D, const float* F5, int n, const uint8_t* masks, cudaStream_t s);
int tdense_head(sc_ctx* ctx, const TcDenseBuf& D, const float* in4, const uint8_t* y, int n, int64_t n_global, const uint8_t* masks, float* loss,
                cudaStream_t s);
int tdense_branch_backward(sc_ctx* ctx, int b, const TcDenseBuf& D, int n, const uint8_t* masks, cudaStream_t s);
int launch_conv1_wgrad(sc_ctx* ctx, const float* patches, const float* dx_planar, int n, int zc, float* gW, cudaStream_t st);

// fused_adam.cu
int fused_export(sc_ctx* ctx, unsigned char* handles);
int fused_attach(sc_ctx* ctx, int rank, int world, const unsigned char* all);
void fused_detach(sc_ctx* ctx);
int fused_allreduce_adam(sc_ctx* ctx, float lr, float b1, float b2, float eps, cudaStream_t st);

// train.cu
int train_forward_backward(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, const float* in4,
                           const uint8_t* y, int64_t n, int64_t n_global, uint64_t seed, const uint8_t* masks,
                           float* loss, cudaStream_t st);
int adam_step(sc_ctx* ctx, float lr, float b1, float b2, float eps, float gscale, float sscale, cudaStream_t st);
int eval_batch(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, const float* in4, const uint8_t* y,
               int64_t n, float* out2, cudaStream_t st);

__device__ __forceinline__ float prelu(float x, float a) { return x > 0.f ? x : a * x; }
// out_layer logits of one voxel (cnn_cort/nets.py:229-231) -> softmax in fp32, in place; returns the argmax on the float32
// probabilities, first maximum wins (np.argmax)
__device__ __forceinline__ int softmax15(float (&z)[15]) {
  float mx = z[0];
#pragma unroll
  for (int c = 1; c < 15; ++c) mx = fmaxf(mx, z[c]);
  float sum = 0.f;
#pragma unroll
  for (int c = 0; c < 15; ++c) { z[c] = expf(z[c] - mx); sum += z[c]; }
  const float inv = 1.f / sum;
  int best = 0;
  float bp = z[0] * inv;
#pragma unroll
  for (int c = 0; c < 15; ++c) {
    z[c] *= inv;
    if (z[c] > bp) { bp = z[c]; best = c; }
  }
  return best;
}
// the softmax / argmax of voxel o go to whichever outputs are set
__device__ __forceinline__ void softmax_store(float (&z)[15], long long o, float* proba, int32_t* label32, uint8_t* label8) {
  const int best = softmax15(z);
  if (proba) {
#pragma unroll
    for (int c = 0; c < 15; ++c) proba[o * 15 + c] = z[c];
  }
  if (label32) label32[o] = best;
  if (label8) label8[o] = (uint8_t)best;
}
// sum_c p_c ln p_c with 0 ln 0 = 0 (minus the entropy in nats): Monte-Carlo dropout evaluates both the per-pass and the
// predictive entropy with this one function, so that one pass gives a mutual information of exactly 0
__device__ __forceinline__ float plogp15(const float (&p)[15]) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 15; ++c) s = p[c] > 0.f ? fmaf(p[c], logf(p[c]), s) : s;
  return s;
}
// split-precision store of 4 consecutive logical columns n..n+3 (n % 4 == 0) of one activation row
__device__ __forceinline__ void store_split4(float* row, int n, float v0, float v1, float v2, float v3) {
  __nv_bfloat16* r = reinterpret_cast<__nv_bfloat16*>(row) + (n >> 6) * 128 + (n & 63);
  const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1), h2 = __float2bfloat16_rn(v2), h3 = __float2bfloat16_rn(v3);
  const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
  const __nv_bfloat16 l2 = __float2bfloat16_rn(v2 - __bfloat162float(h2)), l3 = __float2bfloat16_rn(v3 - __bfloat162float(h3));
  uint2 hp, lp;
  hp.x = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
  hp.y = (uint32_t)__bfloat16_as_ushort(h2) | ((uint32_t)__bfloat16_as_ushort(h3) << 16);
  lp.x = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
  lp.y = (uint32_t)__bfloat16_as_ushort(l2) | ((uint32_t)__bfloat16_as_ushort(l3) << 16);
  *reinterpret_cast<uint2*>(r) = hp;
  *reinterpret_cast<uint2*>(r + 64) = lp;
}
// the same for the 128 B pixel format: 32 bf16 hi | 32 bf16 lo (n < 32)
__device__ __forceinline__ void store_split4_b32(void* px, int n, float v0, float v1, float v2, float v3) {
  __nv_bfloat16* r = reinterpret_cast<__nv_bfloat16*>(px) + n;
  const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1), h2 = __float2bfloat16_rn(v2), h3 = __float2bfloat16_rn(v3);
  const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
  const __nv_bfloat16 l2 = __float2bfloat16_rn(v2 - __bfloat162float(h2)), l3 = __float2bfloat16_rn(v3 - __bfloat162float(h3));
  uint2 hp, lp;
  hp.x = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
  hp.y = (uint32_t)__bfloat16_as_ushort(h2) | ((uint32_t)__bfloat16_as_ushort(h3) << 16);
  lp.x = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
  lp.y = (uint32_t)__bfloat16_as_ushort(l2) | ((uint32_t)__bfloat16_as_ushort(l3) << 16);
  *reinterpret_cast<uint2*>(r) = hp;
  *reinterpret_cast<uint2*>(r + 32) = lp;
}
__device__ __forceinline__ void store_row1(float* row, int n, int split, float v) {
  if (!split) { row[n] = v; return; }
  __nv_bfloat16* r = reinterpret_cast<__nv_bfloat16*>(row) + (n >> 6) * 128 + (n & 63);
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  r[0] = h;
  r[64] = __float2bfloat16_rn(v - __bfloat162float(h));
}
__device__ __forceinline__ void store_row4(float* row, int n, int split, float v0, float v1, float v2, float v3) {
  if (split) store_split4(row, n, v0, v1, v2, v3);
  else *reinterpret_cast<float4*>(row + n) = make_float4(v0, v1, v2, v3);
}
}  // namespace sc
