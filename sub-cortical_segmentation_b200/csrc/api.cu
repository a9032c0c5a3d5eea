// extern "C" surface of libsubcort_b200.so (declared in include/subcort_b200.h).
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <thread>

#include "common.cuh"

namespace sc {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int ensure_ws(Workspace& ws, size_t bytes) {
  if (ws.bytes >= bytes) return SC_OK;
  if (ws.ptr) {
    cudaDeviceSynchronize();
    cudaFree(ws.ptr);
    ws.ptr = nullptr;
    ws.bytes = 0;
  }
  bytes = (bytes + ((size_t)64 << 20) - 1) & ~(((size_t)64 << 20) - 1);
  cudaError_t e = cudaMalloc(&ws.ptr, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("workspace allocation of %zu MiB failed: %s", bytes >> 20, cudaGetErrorString(e));
    ws.ptr = nullptr;
    return SC_ERR_NOMEM;
  }
  ws.bytes = bytes;
  return SC_OK;
}

int ensure_smem_attr(sc_ctx* ctx, const void* kernel, int bytes) {
  for (auto& e : ctx->smem_attr)
    if (e.first == kernel) {
      if (e.second >= bytes) return SC_OK;
      SC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
      e.second = bytes;
      return SC_OK;
    }
  SC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  ctx->smem_attr.emplace_back(kernel, bytes);
  return SC_OK;
}

static int need_weights(sc_ctx* ctx, const char* who) {
  SC_CHECK(ctx != nullptr, SC_ERR_ARG, "%s: null context", who);
  SC_CHECK(ctx->weights_loaded, SC_ERR_STATE, "%s: call sc_load_weights first", who);
  SC_CUDA(cudaSetDevice(ctx->device));
  return SC_OK;
}

// inference entry points call this: re-derive the folded layouts after optimiser steps
static int fresh_weights(sc_ctx* ctx, const char* who, cudaStream_t st) {
  SC_TRY(need_weights(ctx, who));
  if (ctx->derived_dirty) {
    SC_TRY(derive_weights(ctx, st));
    ctx->derived_dirty = false;
  }
  return SC_OK;
}

}  // namespace sc

using namespace sc;

extern "C" {

int sc_version(void) { return 100; }
const char* sc_last_error(void) { return sc::g_err; }

int sc_create(int device, sc_ctx** out) {
  SC_CHECK(out != nullptr, SC_ERR_ARG, "sc_create: null out pointer");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    set_error("sc_create: no CUDA device available (%s); this library has no CPU fallback",
              e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return SC_ERR_CUDA;
  }
  SC_CHECK(device >= 0 && device < count, SC_ERR_ARG, "sc_create: device %d out of range [0,%d)", device, count);
  SC_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SC_CUDA(cudaGetDeviceProperties(&prop, device));
  SC_CHECK(prop.major == 10, SC_ERR_UNSUPPORTED, "sc_create: device %d is sm_%d%d; this library is built for sm_100a only",
           device, prop.major, prop.minor);
  sc_ctx* ctx = new sc_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->off = make_param_off();
  if (ctx->off.total != SC_PARAM_FLOATS) {
    set_error("internal: parameter table has %d floats", ctx->off.total);
    delete ctx;
    return SC_ERR_STATE;
  }
  const size_t pb = sizeof(float) * SC_PARAM_FLOATS;
  SC_CUDA(cudaMalloc(&ctx->params, pb));
  SC_CUDA(cudaMalloc(&ctx->grads, pb));
  SC_CUDA(cudaMalloc(&ctx->adam_m, pb));
  SC_CUDA(cudaMalloc(&ctx->adam_v, pb));
  SC_CUDA(cudaMalloc(&ctx->trainable, SC_PARAM_FLOATS));
  SC_CUDA(cudaMemset(ctx->grads, 0, pb));
  SC_CUDA(cudaMemset(ctx->adam_m, 0, pb));
  SC_CUDA(cudaMemset(ctx->adam_v, 0, pb));
  {
    std::vector<uint8_t> t(SC_PARAM_FLOATS, 1);
    for (int b = 0; b < 3; ++b)
      for (int l = 0; l < 5; ++l)
        for (int k = 2; k < 4; ++k)
          for (int c = 0; c < kConvCout[l]; ++c) t[ctx->off.br[b].bn[l][k] + c] = 0;  // BN mean / inv_std are state
    SC_CUDA(cudaMemcpy(ctx->trainable, t.data(), SC_PARAM_FLOATS, cudaMemcpyHostToDevice));
  }
  SC_CUDA(cudaMalloc(&ctx->d_count, sizeof(int64_t)));
  SC_CUDA(cudaMallocHost(&ctx->h_count, sizeof(int64_t)));
  // the tcgen05 / TMA back-end is the product: a box on which it cannot be brought up is an error, never a silent
  // switch to the SIMT cross-check kernels
  const int tcs = tc_init(ctx);
  if (tcs != SC_OK) {
    sc_destroy(ctx);
    return tcs;
  }
  ctx->gemm_backend = 1;
  *out = ctx;
  return SC_OK;
}

int sc_destroy(sc_ctx* ctx) {
  if (!ctx) return SC_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  tc_destroy(ctx);
  fused_detach(ctx);
  cudaFree(ctx->params); cudaFree(ctx->grads); cudaFree(ctx->adam_m); cudaFree(ctx->adam_v);
  cudaFree(ctx->trainable); cudaFree(ctx->derived); cudaFree(ctx->ws.ptr); cudaFree(ctx->ws_train.ptr); cudaFree(ctx->ws_fit.ptr); cudaFree(ctx->ws_eval.ptr); cudaFree(ctx->ws_reg.ptr);
  for (auto& g : ctx->train_graphs) cudaGraphExecDestroy(g.exec);
  for (int i = 0; i < 2; ++i) if (ctx->train_side[i]) cudaStreamDestroy(ctx->train_side[i]);
  for (int i = 0; i < 8; ++i) if (ctx->train_ev[i]) cudaEventDestroy(ctx->train_ev[i]);
  cudaFree(ctx->d_count); cudaFreeHost(ctx->h_count); cudaFree(ctx->train_consts); cudaFree(ctx->tc_timing_buf); cudaFree(ctx->train_panels); cudaFree(ctx->train_dense_w);
  for (auto& ev : ctx->prof_live) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
  for (auto& ev : ctx->prof_free) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
  if (ctx->h_slab_cnt) { cudaFreeHost(ctx->h_slab_cnt); cudaEventDestroy(ctx->compact_ev); }
  cudaFree(ctx->tile_flags);
  cudaFree(ctx->mc_w);
  if (ctx->h_reg) cudaFreeHost(ctx->h_reg);
  for (int i = 0; i < 64; ++i) if (ctx->atlas_chunk_ev[i]) cudaEventDestroy(ctx->atlas_chunk_ev[i]);
  if (ctx->copy_stream) { cudaStreamDestroy(ctx->copy_stream); cudaEventDestroy(ctx->copy_ev[0]); cudaEventDestroy(ctx->copy_ev[1]); }
  delete ctx;
  return SC_OK;
}

int sc_set_option(sc_ctx* ctx, const char* key, int64_t value) {
  SC_CHECK(ctx && key, SC_ERR_ARG, "sc_set_option: null argument");
  if (!strcmp(key, "gemm")) {
    SC_CHECK(value == 0 || value == 1, SC_ERR_ARG, "sc_set_option: gemm must be 0 (SIMT) or 1 (tcgen05)");
    SC_CHECK(value == 0 || ctx->tc_state != nullptr, SC_ERR_UNSUPPORTED, "sc_set_option: tcgen05 back-end unavailable");
    ctx->gemm_backend = (int)value;
    return SC_OK;
  }
  if (!strcmp(key, "tc_timing")) {   // value = ProfClass index to instrument, -1 = off
    ctx->tc_timing_cls = (int)value;
    if (value >= 0 && !ctx->tc_timing_buf) SC_CUDA(cudaMalloc(&ctx->tc_timing_buf, sizeof(unsigned long long) * 8 * 1024));
    return SC_OK;
  }
  if (!strcmp(key, "tc_skip")) {
    ctx->tc_skip = value != 0;
    return SC_OK;
  }
  if (!strcmp(key, "tc_compact")) {
    ctx->tc_compact = value != 0;
    return SC_OK;
  }
  if (!strcmp(key, "gather_ctas_per_sm")) {
    SC_CHECK(value >= 0 && value <= 32, SC_ERR_ARG, "sc_set_option: gather_ctas_per_sm must be 0..32");
    ctx->gather_ctas_per_sm = (int)value;
    return SC_OK;
  }
  if (!strcmp(key, "train_graph")) {
    ctx->train_graph_on = value != 0;
    return SC_OK;
  }
  if (!strcmp(key, "train_fused_stats") || !strcmp(key, "train_wgrad_mn")) {     // captured graphs hold the launch sequence of the setting they were captured under
    int& opt = !strcmp(key, "train_fused_stats") ? ctx->train_fused_stats : ctx->train_wgrad_mn;
    if ((value != 0) != (opt != 0)) {
      for (auto& g : ctx->train_graphs) cudaGraphExecDestroy(g.exec);
      ctx->train_graphs.clear();
    }
    opt = value != 0;
    return SC_OK;
  }
  if (!strcmp(key, "profile")) {
    ctx->profile = value != 0;
    return SC_OK;
  }
  if (!strcmp(key, "chunk_voxels")) {
    SC_CHECK(value >= 1024, SC_ERR_ARG, "sc_set_option: chunk_voxels must be >= 1024");
    ctx->chunk_voxels = value;
    return SC_OK;
  }
  set_error("sc_set_option: unknown key '%s'", key);
  return SC_ERR_ARG;
}

int64_t sc_get_counter(sc_ctx* ctx, const char* key) {
  if (!ctx || !key) return -1;
  if (!strncmp(key, "tc_timing:", 10) && ctx->tc_timing_buf) {   // "tc_timing:<index>" -> one debug counter
    const int i = atoi(key + 10);
    unsigned long long v = 0;
    if (i < 0 || i >= 8 * 1024) return -1;
    cudaDeviceSynchronize();
    cudaMemcpy(&v, ctx->tc_timing_buf + i, sizeof(v), cudaMemcpyDeviceToHost);
    return (int64_t)v;
  }
  if (!strncmp(key, "reg_iters:", 10)) {   // accepted steps per level of the last registration: 0..3 affine, 4..6 FFD
    const int i = atoi(key + 10);
    return i >= 0 && i < 8 ? ctx->reg_iters[i] : -1;
  }
  if (!strcmp(key, "launches")) return ctx->launches;
  if (!strcmp(key, "gemm")) return ctx->gemm_backend;
  if (!strcmp(key, "adam_t")) return ctx->adam_t;
  if (!strcmp(key, "workspace_bytes")) return (int64_t)ctx->ws.bytes;
  return -1;
}

static const char* kProfNames[PC_COUNT] = {"gather", "nonzero", "scatter", "patch_branch", "conv1", "conv2", "conv3",
                                           "conv4", "conv5", "gemm_d1", "gemm_fc1", "gemm_fc2", "atlas", "out_softmax", "pool",
                                           "train_fwd", "train_bwd", "adam", "evaluate", "register", "mc"};
}  // extern "C"
namespace sc { const char* prof_class_name(int cls) { return cls >= 0 && cls < PC_COUNT ? kProfNames[cls] : "subcort"; } }
extern "C" {
int sc_profile_classes(void) { return PC_COUNT; }
const char* sc_profile_name(int cls) { return cls >= 0 && cls < PC_COUNT ? kProfNames[cls] : ""; }
int sc_profile_read(sc_ctx* ctx, double* ms_out, int64_t* launches_out, int n) {
  SC_CHECK(ctx && ms_out && launches_out && n >= PC_COUNT, SC_ERR_ARG, "sc_profile_read: bad argument");
  SC_CUDA(cudaSetDevice(ctx->device));
  SC_CUDA(cudaDeviceSynchronize());
  for (int i = 0; i < n; ++i) { ms_out[i] = 0.0; launches_out[i] = 0; }
  for (auto& ev : ctx->prof_live) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) { ms_out[ev.cls] += ms; launches_out[ev.cls]++; }
    ctx->prof_free.push_back(ev);
  }
  cudaGetLastError();
  ctx->prof_live.clear();
  return SC_OK;
}

int sc_load_weights(sc_ctx* ctx, const float* blob_host, int64_t n_floats) {
  SC_CHECK(ctx && blob_host, SC_ERR_ARG, "sc_load_weights: null argument");
  SC_CHECK(n_floats == SC_PARAM_FLOATS, SC_ERR_ARG, "sc_load_weights: expected %d floats, got %lld", SC_PARAM_FLOATS,
           (long long)n_floats);
  SC_CUDA(cudaSetDevice(ctx->device));
  SC_CUDA(cudaMemcpy(ctx->params, blob_host, sizeof(float) * SC_PARAM_FLOATS, cudaMemcpyHostToDevice));
  SC_TRY(derive_weights(ctx, nullptr));
  ctx->weights_loaded = true;
  ctx->derived_dirty = false;
  return SC_OK;
}

int sc_get_params(sc_ctx* ctx, float* blob_host, int64_t n_floats) {
  SC_TRY(need_weights(ctx, "sc_get_params"));
  SC_CHECK(blob_host && n_floats == SC_PARAM_FLOATS, SC_ERR_ARG, "sc_get_params: bad buffer");
  SC_CUDA(cudaDeviceSynchronize());
  SC_CUDA(cudaMemcpy(blob_host, ctx->params, sizeof(float) * SC_PARAM_FLOATS, cudaMemcpyDeviceToHost));
  return SC_OK;
}

static int check_dims(const int32_t* dims, const char* who) {
  SC_CHECK(dims && dims[0] > 0 && dims[1] > 0 && dims[2] > 0, SC_ERR_ARG, "%s: bad volume dims", who);
  SC_CHECK((int64_t)dims[0] * dims[1] * dims[2] < (1ll << 31), SC_ERR_ARG, "%s: volume too large", who);
  return SC_OK;
}

int sc_nonzero_coords(sc_ctx* ctx, const void* vol_dev, int elem_bytes, const int32_t dims[3], int32_t* xyz_dev,
                      int64_t capacity, int64_t* n_out_host, void* stream) {
  SC_CHECK(ctx && vol_dev, SC_ERR_ARG, "sc_nonzero_coords: null argument");
  SC_TRY(check_dims(dims, "sc_nonzero_coords"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return launch_nonzero(ctx, vol_dev, elem_bytes, dims, xyz_dev, capacity, n_out_host, (cudaStream_t)stream);
}

int sc_dilate_mask(sc_ctx* ctx, const uint8_t* mask_dev, const int32_t dims[3], int iterations, uint8_t* out_dev, void* stream) {
  SC_CHECK(ctx && mask_dev && out_dev && mask_dev != out_dev, SC_ERR_ARG, "sc_dilate_mask: bad argument");
  SC_TRY(check_dims(dims, "sc_dilate_mask"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return launch_dilate(ctx, mask_dev, dims, iterations, out_dev, (cudaStream_t)stream);
}

int sc_import_volume(sc_ctx* ctx, const void* src_dev, int elem_bytes, const int32_t dims[3], int channels, void* dst_dev, void* stream) {
  SC_CHECK(ctx && src_dev && dst_dev && src_dev != dst_dev && channels >= 1, SC_ERR_ARG, "sc_import_volume: bad argument");
  SC_TRY(check_dims(dims, "sc_import_volume"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return import_volume(ctx, src_dev, elem_bytes, dims, channels, dst_dev, (cudaStream_t)stream);
}

int sc_upload_volume_box(sc_ctx* ctx, const void* src_host, int elem_bytes, const int32_t dims[3], int channels, int fortran_order,
                         const int32_t box[6], void* staging_dev, void* dst_dev, void* stream) {
  SC_CHECK(ctx && src_host && dst_dev && box && channels >= 1, SC_ERR_ARG, "sc_upload_volume_box: bad argument");
  SC_CHECK(elem_bytes == 1 || elem_bytes == 2 || elem_bytes == 4 || elem_bytes == 8, SC_ERR_ARG, "sc_upload_volume_box: elem_bytes must be 1, 2, 4 or 8");
  SC_TRY(check_dims(dims, "sc_upload_volume_box"));
  SC_CHECK(box[0] >= 0 && box[0] < box[1] && box[1] <= dims[0] && box[2] >= 0 && box[2] < box[3] && box[3] <= dims[1] &&
           box[4] >= 0 && box[4] < box[5] && box[5] <= dims[2], SC_ERR_ARG, "sc_upload_volume_box: empty box or box outside the volume");
  SC_CUDA(cudaSetDevice(ctx->device));
  return upload_volume_box(ctx, src_host, elem_bytes, dims, channels, fortran_order, box, staging_dev, dst_dev, (cudaStream_t)stream);
}

int sc_normalise_volume(sc_ctx* ctx, const void* vol_dev, int dtype, const int32_t dims[3], float* out_dev, double* mean_std_host, void* stream) {
  SC_CHECK(ctx && vol_dev && (out_dev || mean_std_host), SC_ERR_ARG, "sc_normalise_volume: bad argument");
  SC_TRY(check_dims(dims, "sc_normalise_volume"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return normalise_volume(ctx, vol_dev, dtype, dims, out_dev, mean_std_host, (cudaStream_t)stream);
}

int sc_candidate_mask(sc_ctx* ctx, const void* vol_dev, int dtype, const int32_t dims[3], uint8_t* mask_dev, void* stream) {
  SC_CHECK(ctx && vol_dev && mask_dev, SC_ERR_ARG, "sc_candidate_mask: bad argument");
  SC_TRY(check_dims(dims, "sc_candidate_mask"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return candidate_mask(ctx, vol_dev, dtype, dims, mask_dev, (cudaStream_t)stream);
}

int sc_mask_bbox(sc_ctx* ctx, const uint8_t* mask_dev, const int32_t dims[3], int32_t box_host[6], int64_t* count_host, void* stream) {
  SC_CHECK(ctx && mask_dev && box_host, SC_ERR_ARG, "sc_mask_bbox: bad argument");
  SC_TRY(check_dims(dims, "sc_mask_bbox"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return mask_bbox(ctx, mask_dev, dims, box_host, count_host, (cudaStream_t)stream);
}

int sc_post_process(sc_ctx* ctx, const uint8_t* seg_dev, const uint8_t* mask_dev, const int32_t dims[3], uint8_t* out_dev, void* stream) {
  SC_CHECK(ctx && seg_dev && mask_dev && out_dev && out_dev != seg_dev, SC_ERR_ARG, "sc_post_process: bad argument");
  SC_TRY(check_dims(dims, "sc_post_process"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return post_process(ctx, seg_dev, mask_dev, dims, out_dev, (cudaStream_t)stream);
}

int sc_evaluate_segmentation(sc_ctx* ctx, const uint8_t* seg_dev, const uint8_t* ref_dev, const int32_t dims[3], const double spacing[3],
                             sc_structure_metrics* metrics_host, int64_t* confusion_host, void* stream) {
  SC_CHECK(ctx && seg_dev && ref_dev && spacing && metrics_host, SC_ERR_ARG, "sc_evaluate_segmentation: null argument");
  SC_TRY(check_dims(dims, "sc_evaluate_segmentation"));
  for (int i = 0; i < 3; ++i)
    SC_CHECK(isfinite(spacing[i]) && spacing[i] > 0.0, SC_ERR_ARG, "sc_evaluate_segmentation: spacing[%d] = %g is not a finite positive number",
             i, spacing[i]);
  SC_CUDA(cudaSetDevice(ctx->device));
  return evaluate_segmentation(ctx, seg_dev, ref_dev, dims, spacing, metrics_host, confusion_host, (cudaStream_t)stream);
}

// registration arguments: a volume of dims >= 8 and a finite, non-singular voxel -> mm matrix
static int check_reg_volume(const void* dev, const int32_t* dims, const char* who, const char* name) {
  SC_CHECK(dev != nullptr, SC_ERR_ARG, "%s: %s is NULL", who, name);
  SC_CHECK(dims != nullptr, SC_ERR_ARG, "%s: %s dims are NULL", who, name);
  for (int i = 0; i < 3; ++i)
    SC_CHECK(dims[i] >= 8, SC_ERR_ARG, "%s: %s dims[%d] = %d is below 8", who, name, i, dims[i]);
  SC_CHECK((int64_t)dims[0] * dims[1] * dims[2] < (1ll << 31), SC_ERR_ARG, "%s: %s volume too large", who, name);
  return SC_OK;
}
static int check_matrix(const double* m, const char* who, const char* name) {
  SC_CHECK(m != nullptr, SC_ERR_ARG, "%s: %s is NULL", who, name);
  for (int i = 0; i < 16; ++i) SC_CHECK(isfinite(m[i]), SC_ERR_ARG, "%s: %s[%d] is not finite", who, name, i);
  const double det = m[0] * (m[5] * m[10] - m[6] * m[9]) - m[1] * (m[4] * m[10] - m[6] * m[8]) + m[2] * (m[4] * m[9] - m[5] * m[8]);
  SC_CHECK(fabs(det) > 1e-12, SC_ERR_ARG, "%s: %s is singular", who, name);
  return SC_OK;
}

int sc_ffd_grid_dims(const int32_t ref_dims[3], int32_t grid_dims_out[3]) {
  SC_CHECK(ref_dims && grid_dims_out, SC_ERR_ARG, "sc_ffd_grid_dims: null argument");
  for (int i = 0; i < 3; ++i) SC_CHECK(ref_dims[i] >= 8, SC_ERR_ARG, "sc_ffd_grid_dims: ref_dims[%d] = %d is below 8", i, ref_dims[i]);
  ffd_grid_dims(ref_dims, grid_dims_out);
  return SC_OK;
}

int sc_register_affine(sc_ctx* ctx, const float* ref_dev, const int32_t ref_dims[3], const double ref_vox2mm[16], const float* flo_dev,
                       const int32_t flo_dims[3], const double flo_vox2mm[16], double affine_out[16], void* stream) {
  const char* who = "sc_register_affine";
  SC_CHECK(ctx && affine_out, SC_ERR_ARG, "%s: null context or affine_out", who);
  SC_TRY(check_reg_volume(ref_dev, ref_dims, who, "ref_dev"));
  SC_TRY(check_reg_volume(flo_dev, flo_dims, who, "flo_dev"));
  SC_TRY(check_matrix(ref_vox2mm, who, "ref_vox2mm"));
  SC_TRY(check_matrix(flo_vox2mm, who, "flo_vox2mm"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return register_affine(ctx, ref_dev, ref_dims, ref_vox2mm, flo_dev, flo_dims, flo_vox2mm, affine_out, (cudaStream_t)stream);
}

int sc_register_ffd(sc_ctx* ctx, const float* ref_dev, const int32_t ref_dims[3], const double ref_vox2mm[16], const float* flo_dev,
                    const int32_t flo_dims[3], const double flo_vox2mm[16], const double affine[16], float* grid_dev, void* stream) {
  const char* who = "sc_register_ffd";
  SC_CHECK(ctx && grid_dev, SC_ERR_ARG, "%s: null context or grid_dev", who);
  SC_TRY(check_reg_volume(ref_dev, ref_dims, who, "ref_dev"));
  SC_TRY(check_reg_volume(flo_dev, flo_dims, who, "flo_dev"));
  SC_TRY(check_matrix(ref_vox2mm, who, "ref_vox2mm"));
  SC_TRY(check_matrix(flo_vox2mm, who, "flo_vox2mm"));
  SC_TRY(check_matrix(affine, who, "affine"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return register_ffd(ctx, ref_dev, ref_dims, ref_vox2mm, flo_dev, flo_dims, flo_vox2mm, affine, grid_dev, (cudaStream_t)stream);
}

int sc_warp_volume(sc_ctx* ctx, const float* flo_dev, const int32_t flo_dims[3], int channels, const double flo_vox2mm[16],
                   const double affine[16], const float* grid_dev, const int32_t ref_dims[3], const double ref_vox2mm[16], float* out_dev,
                   void* stream) {
  const char* who = "sc_warp_volume";
  SC_CHECK(ctx && out_dev, SC_ERR_ARG, "%s: null context or out_dev", who);
  SC_CHECK(channels == 1 || channels == 15, SC_ERR_ARG, "%s: channels = %d (1 or 15)", who, channels);
  SC_TRY(check_reg_volume(flo_dev, flo_dims, who, "flo_dev"));
  SC_TRY(check_reg_volume(out_dev, ref_dims, who, "out_dev"));
  SC_TRY(check_matrix(flo_vox2mm, who, "flo_vox2mm"));
  SC_TRY(check_matrix(ref_vox2mm, who, "ref_vox2mm"));
  SC_TRY(check_matrix(affine, who, "affine"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return warp_volume(ctx, flo_dev, flo_dims, channels, flo_vox2mm, affine, grid_dev, ref_dims, ref_vox2mm, out_dev, (cudaStream_t)stream);
}

int sc_register_objective(sc_ctx* ctx, const float* ref_dev, const int32_t ref_dims[3], const double ref_vox2mm[16], const float* flo_dev,
                          const int32_t flo_dims[3], const double flo_vox2mm[16], const double affine[16], const float* grid_dev,
                          double value_out[3], double* affine_grad_host, float* grid_grad_dev, void* stream) {
  const char* who = "sc_register_objective";
  SC_CHECK(ctx && value_out, SC_ERR_ARG, "%s: null context or value_out", who);
  SC_CHECK(grid_dev || !grid_grad_dev, SC_ERR_ARG, "%s: grid_grad_dev needs grid_dev", who);
  SC_TRY(check_reg_volume(ref_dev, ref_dims, who, "ref_dev"));
  SC_TRY(check_reg_volume(flo_dev, flo_dims, who, "flo_dev"));
  SC_TRY(check_matrix(ref_vox2mm, who, "ref_vox2mm"));
  SC_TRY(check_matrix(flo_vox2mm, who, "flo_vox2mm"));
  SC_TRY(check_matrix(affine, who, "affine"));
  SC_CUDA(cudaSetDevice(ctx->device));
  double ga[12];
  SC_TRY(register_objective(ctx, ref_dev, ref_dims, ref_vox2mm, flo_dev, flo_dims, flo_vox2mm, affine, grid_dev, value_out,
                            affine_grad_host ? ga : nullptr, grid_grad_dev, (cudaStream_t)stream));
  if (affine_grad_host) memcpy(affine_grad_host, ga, sizeof(ga));   // uncentred: the objective's sums use c = 0
  return SC_OK;
}

int sc_prior_mask(sc_ctx* ctx, const float* priors_dev, const int32_t dims[3], int iterations, float* mask_dev, void* stream) {
  SC_CHECK(ctx && priors_dev && mask_dev, SC_ERR_ARG, "sc_prior_mask: null argument");
  SC_CHECK(iterations >= 0, SC_ERR_ARG, "sc_prior_mask: iterations = %d is negative", iterations);
  SC_TRY(check_dims(dims, "sc_prior_mask"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return prior_mask(ctx, priors_dev, dims, iterations, mask_dev, (cudaStream_t)stream);
}

int sc_gather_patches(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3], const float* atlas_dev, int bg_fix,
                      const int32_t* xyz_dev, int64_t n, float* axial_dev, float* coronal_dev, float* saggital_dev,
                      float* atlas_out_dev, void* stream) {
  SC_CHECK(ctx && vol_dev && (xyz_dev || n == 0) && n >= 0, SC_ERR_ARG, "sc_gather_patches: bad argument");
  SC_TRY(check_dims(dims, "sc_gather_patches"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return launch_gather(ctx, vol_dev, dims, atlas_dev, bg_fix, xyz_dev, n, axial_dev, coronal_dev, saggital_dev,
                       atlas_out_dev, (cudaStream_t)stream);
}

int sc_gather_center_labels(sc_ctx* ctx, const uint8_t* labels_dev, const int32_t dims[3], const int32_t* xyz_dev,
                            int64_t n, uint8_t* y_dev, void* stream) {
  SC_CHECK(ctx && labels_dev && (xyz_dev || n == 0) && (y_dev || n == 0) && n >= 0, SC_ERR_ARG, "sc_gather_center_labels: bad argument");
  SC_TRY(check_dims(dims, "sc_gather_center_labels"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return launch_center_labels(ctx, labels_dev, dims, xyz_dev, n, y_dev, (cudaStream_t)stream);
}

int sc_gather_samples(sc_ctx* ctx, const sc_scan* scans_dev, int n_scans, const int32_t* samples_dev, const float* atlas_rows_dev,
                      const uint8_t* labels_dev, const int64_t* idx_dev, int64_t n, float* axial_dev, float* coronal_dev,
                      float* saggital_dev, float* atlas_out_dev, uint8_t* y_out_dev, void* stream) {
  SC_CHECK(ctx && n >= 0 && n_scans >= 0, SC_ERR_ARG, "sc_gather_samples: null context or negative count");
  SC_CHECK(!atlas_out_dev || atlas_rows_dev, SC_ERR_ARG, "sc_gather_samples: atlas output requested without atlas rows");
  SC_CHECK(!y_out_dev || labels_dev, SC_ERR_ARG, "sc_gather_samples: label output requested without labels");
  if (n == 0) return SC_OK;
  SC_CHECK(scans_dev && n_scans > 0 && samples_dev, SC_ERR_ARG, "sc_gather_samples: missing scan list or sample table");
  SC_CHECK(((uintptr_t)samples_dev & 15) == 0, SC_ERR_ARG, "sc_gather_samples: sample table not 16-byte aligned");
  SC_CUDA(cudaSetDevice(ctx->device));
  return launch_gather_samples(ctx, scans_dev, n_scans, samples_dev, atlas_rows_dev, labels_dev, idx_dev, n, axial_dev,
                               coronal_dev, saggital_dev, atlas_out_dev, y_out_dev, (cudaStream_t)stream);
}

int sc_forward(sc_ctx* ctx, const float* in1_dev, const float* in2_dev, const float* in3_dev, const float* in4_dev,
               int64_t n, float* proba_dev, int32_t* label_dev, void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_forward", (cudaStream_t)stream));
  SC_CHECK(n >= 0, SC_ERR_ARG, "sc_forward: negative batch");
  if (n == 0) return SC_OK;
  SC_CHECK(in1_dev && in2_dev && in3_dev && in4_dev, SC_ERR_ARG, "sc_forward: null input");
  return forward_patches(ctx, in1_dev, in2_dev, in3_dev, in4_dev, n, proba_dev, label_dev, (cudaStream_t)stream);
}

int sc_forward_host(sc_ctx* ctx, const float* in1_host, const float* in2_host, const float* in3_host,
                    const float* in4_host, int64_t n, float* proba_host, int32_t* label_host, void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_forward_host", (cudaStream_t)stream));
  SC_CHECK(n >= 0, SC_ERR_ARG, "sc_forward_host: negative batch");
  if (n == 0) return SC_OK;
  SC_CHECK(in1_host && in2_host && in3_host && in4_host, SC_ERR_ARG, "sc_forward_host: null input");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t chunk = 32768;
  const int64_t cmax = n < chunk ? n : chunk;
  const size_t pb = (size_t)cmax * 1024 * sizeof(float);
  const size_t bytes = 3 * pb + (size_t)cmax * (15 + 15 + 1) * sizeof(float);
  SC_TRY(ensure_ws(ctx->ws_train, bytes));  // staging lives in the second arena; forward_patches uses ctx->ws
  char* base = reinterpret_cast<char*>(ctx->ws_train.ptr);
  float* d_in[3] = {reinterpret_cast<float*>(base), reinterpret_cast<float*>(base + pb), reinterpret_cast<float*>(base + 2 * pb)};
  float* d_at = reinterpret_cast<float*>(base + 3 * pb);
  float* d_pr = d_at + cmax * 15;
  int32_t* d_lb = reinterpret_cast<int32_t*>(d_pr + cmax * 15);
  const float* h_in[3] = {in1_host, in2_host, in3_host};
  for (int64_t s = 0; s < n; s += chunk) {
    const int64_t m = n - s < chunk ? n - s : chunk;
    for (int b = 0; b < 3; ++b)
      SC_CUDA(cudaMemcpyAsync(d_in[b], h_in[b] + s * 1024, (size_t)m * 4096, cudaMemcpyHostToDevice, st));
    SC_CUDA(cudaMemcpyAsync(d_at, in4_host + s * 15, (size_t)m * 60, cudaMemcpyHostToDevice, st));
    SC_TRY(forward_patches(ctx, d_in[0], d_in[1], d_in[2], d_at, m, d_pr, d_lb, st));
    if (proba_host) SC_CUDA(cudaMemcpyAsync(proba_host + s * 15, d_pr, (size_t)m * 60, cudaMemcpyDeviceToHost, st));
    if (label_host) SC_CUDA(cudaMemcpyAsync(label_host + s, d_lb, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
  }
  SC_CUDA(cudaStreamSynchronize(st));
  return SC_OK;
}

int sc_forward_from_volume(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3], const float* atlas_dev,
                           const int32_t* xyz_dev, int64_t n, float* proba_dev, int32_t* label_dev, void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_forward_from_volume", (cudaStream_t)stream));
  SC_CHECK(n >= 0, SC_ERR_ARG, "sc_forward_from_volume: negative batch");
  if (n == 0) return SC_OK;
  SC_CHECK(vol_dev && atlas_dev && xyz_dev, SC_ERR_ARG, "sc_forward_from_volume: null input");
  SC_TRY(check_dims(dims, "sc_forward_from_volume"));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t chunk = 32768;
  const int64_t cmax = n < chunk ? n : chunk;
  const size_t pb = (size_t)cmax * 1024 * sizeof(float);
  SC_TRY(ensure_ws(ctx->ws_train, 3 * pb + (size_t)cmax * 15 * sizeof(float)));
  char* base = reinterpret_cast<char*>(ctx->ws_train.ptr);
  float* d_in[3] = {reinterpret_cast<float*>(base), reinterpret_cast<float*>(base + pb), reinterpret_cast<float*>(base + 2 * pb)};
  float* d_at = reinterpret_cast<float*>(base + 3 * pb);
  for (int64_t s = 0; s < n; s += chunk) {
    const int64_t m = n - s < chunk ? n - s : chunk;
    SC_TRY(launch_gather(ctx, vol_dev, dims, atlas_dev, 1, xyz_dev + s * 3, m, d_in[0], d_in[1], d_in[2], d_at, st));
    SC_TRY(forward_patches(ctx, d_in[0], d_in[1], d_in[2], d_at, m, proba_dev ? proba_dev + s * 15 : nullptr,
                           label_dev ? label_dev + s : nullptr, st));
  }
  return SC_OK;
}

int sc_segment_volume(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3], const float* atlas_dev,
                      const int32_t* box, const uint8_t* cand_mask_dev, uint8_t* label_vol_dev, float* proba_vol_dev,
                      void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_segment_volume", (cudaStream_t)stream));
  SC_CHECK(vol_dev && atlas_dev && (label_vol_dev || proba_vol_dev), SC_ERR_ARG, "sc_segment_volume: null argument");
  SC_TRY(check_dims(dims, "sc_segment_volume"));
  return segment_volume(ctx, vol_dev, dims, atlas_dev, box, cand_mask_dev, label_vol_dev, proba_vol_dev, (cudaStream_t)stream);
}

int sc_segment_volume_mc(sc_ctx* ctx, const float* vol_dev, const int32_t dims[3], const float* atlas_dev, const int32_t* box,
                         const uint8_t* cand_mask_dev, int samples, uint64_t seed, uint8_t* label_vol_dev, float* proba_vol_dev,
                         float* entropy_vol_dev, float* mi_vol_dev, void* stream) {
  const char* who = "sc_segment_volume_mc";
  SC_TRY(fresh_weights(ctx, who, (cudaStream_t)stream));
  SC_CHECK(vol_dev, SC_ERR_ARG, "%s: vol_dev is NULL", who);
  SC_CHECK(atlas_dev, SC_ERR_ARG, "%s: atlas_dev is NULL", who);
  SC_CHECK(label_vol_dev || proba_vol_dev || entropy_vol_dev || mi_vol_dev, SC_ERR_ARG,
           "%s: label_vol, proba_vol, entropy_vol and mi_vol are all NULL", who);
  SC_CHECK(samples >= 1 && samples <= 1024, SC_ERR_ARG, "%s: samples = %d is outside [1, 1024]", who, samples);
  SC_CHECK(ctx->gemm_backend == 1, SC_ERR_ARG, "%s: Monte-Carlo dropout runs on the tcgen05 back-end only (gemm = %d)", who,
           ctx->gemm_backend);
  SC_TRY(check_dims(dims, who));
  if (box)
    SC_CHECK(box[0] >= 0 && box[1] <= dims[0] && box[2] >= 0 && box[3] <= dims[1] && box[4] >= 0 && box[5] <= dims[2], SC_ERR_ARG,
             "%s: box {%d,%d,%d,%d,%d,%d} outside the volume", who, box[0], box[1], box[2], box[3], box[4], box[5]);
  const McArgs mc = {samples, seed, entropy_vol_dev, mi_vol_dev};
  return segment_volume(ctx, vol_dev, dims, atlas_dev, box, cand_mask_dev, label_vol_dev, proba_vol_dev, (cudaStream_t)stream, &mc);
}

int sc_atlas_ready_event(sc_ctx* ctx, void* cuda_event) {
  SC_CHECK(ctx, SC_ERR_ARG, "sc_atlas_ready_event: null context");
  ctx->atlas_ready = (cudaEvent_t)cuda_event;
  ctx->atlas_chunks = 0;
  return SC_OK;
}

int sc_segment_volume_host(sc_ctx* ctx, const float* vol_host, const int32_t dims[3], const float* atlas_host,
                           const int32_t* box, const uint8_t* cand_mask_host, uint8_t* label_vol_host,
                           float* proba_vol_host, void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_segment_volume_host", (cudaStream_t)stream));
  SC_CHECK(vol_host && atlas_host && (label_vol_host || proba_vol_host), SC_ERR_ARG, "sc_segment_volume_host: null argument");
  SC_TRY(check_dims(dims, "sc_segment_volume_host"));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nvox = (size_t)dims[0] * dims[1] * dims[2];
  const size_t vb = (nvox * 4 + 255) & ~(size_t)255, ab = (nvox * 60 + 255) & ~(size_t)255, mb = (nvox + 255) & ~(size_t)255;
  const size_t pb = proba_vol_host ? ab : 0;
  SC_TRY(ensure_ws(ctx->ws_train, vb + ab + 2 * mb + pb));
  char* base = reinterpret_cast<char*>(ctx->ws_train.ptr);
  float* d_vol = reinterpret_cast<float*>(base);
  float* d_atlas = reinterpret_cast<float*>(base + vb);
  uint8_t* d_mask = reinterpret_cast<uint8_t*>(base + vb + ab);
  uint8_t* d_lab = d_mask + mb;
  float* d_proba = proba_vol_host ? reinterpret_cast<float*>(base + vb + ab + 2 * mb) : nullptr;
  std::atomic<int> atlas_recorded(0), upload_err(0);
  std::thread uploader;
  // on every return path: join the helper, drop the per-call upload state from the context (it points at this frame),
  // and on an error path wait for the copies that may still be reading the caller's buffers
  struct Joiner {
    std::thread& t; sc_ctx* ctx; cudaStream_t st; bool ok;
    ~Joiner() {
      if (t.joinable()) t.join();
      ctx->atlas_recorded = nullptr; ctx->atlas_chunks = 0; ctx->atlas_ready = nullptr;
      if (!ok) {
        if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamSynchronize(st);
        cudaGetLastError();
      }
    }
  } joiner{uploader, ctx, st, false};
  // the atlas (15 floats per voxel, 94 % of the upload) is first needed after the conv phase: upload it on a side
  // stream so that the copy engine works while the conv kernels run
  if (!ctx->copy_stream) {
    SC_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) SC_CUDA(cudaEventCreateWithFlags(&ctx->copy_ev[i], cudaEventDisableTiming));
  }
  // the volume and the mask go first: the conv phase waits for them, and host-to-device copies of different streams
  // are served in issue order -- queued behind the 1 GB atlas they would delay the first kernel by ~20 ms
  SC_CUDA(cudaMemcpyAsync(d_vol, vol_host, nvox * 4, cudaMemcpyHostToDevice, st));
  if (cand_mask_host) SC_CUDA(cudaMemcpyAsync(d_mask, cand_mask_host, nvox, cudaMemcpyHostToDevice, st));
  SC_CUDA(cudaEventRecord(ctx->copy_ev[0], st));                       // also: earlier work on `st` may still read the staging buffers
  SC_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev[0], 0));
  {
    // in chunks of x-planes (at most 64), each with its own event: the first slab of phase 2 can start as soon as its
    // planes have arrived, however slow the rest of the upload is under the memory traffic of the kernels
    const size_t plane_b = (size_t)dims[1] * dims[2] * 60;
    int cnx = (dims[0] + 63) / 64;
    const int slab_nx = (int)(ctx->chunk_voxels / ((int64_t)dims[1] * dims[2]));
    if (cnx < slab_nx) cnx = slab_nx;
    if (cnx < 1) cnx = 1;
    const int nch = (dims[0] + cnx - 1) / cnx;
    for (int i = 0; i < nch; ++i)
      if (!ctx->atlas_chunk_ev[i]) SC_CUDA(cudaEventCreateWithFlags(&ctx->atlas_chunk_ev[i], cudaEventDisableTiming));
    ctx->atlas_chunks = nch; ctx->atlas_chunk_nx = cnx;
    ctx->atlas_ready = ctx->atlas_chunk_ev[nch - 1];
    auto upload = [=, &atlas_recorded, &upload_err]() {
      cudaSetDevice(ctx->device);
      for (int i = 0; i < nch; ++i) {
        const int x0 = i * cnx, nx = dims[0] - x0 < cnx ? dims[0] - x0 : cnx;
        cudaError_t e = cudaMemcpyAsync(reinterpret_cast<char*>(d_atlas) + (size_t)x0 * plane_b,
                                        reinterpret_cast<const char*>(atlas_host) + (size_t)x0 * plane_b, (size_t)nx * plane_b,
                                        cudaMemcpyHostToDevice, ctx->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(ctx->atlas_chunk_ev[i], ctx->copy_stream);
        if (e != cudaSuccess) upload_err.store((int)e);
        atlas_recorded.store(i + 1, std::memory_order_release);      // (on an error too: the consumer must not spin forever)
      }
    };
    // pinned (or registered) host memory: the copies are asynchronous, issue them right here.  Pageable memory: every
    // cudaMemcpyAsync blocks its caller while the driver stages the data, so a helper thread issues them and this
    // thread goes on to launch the conv phase -- the upload still overlaps the kernels
    cudaPointerAttributes pa;
    const bool pageable = cudaPointerGetAttributes(&pa, atlas_host) != cudaSuccess || pa.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    bool threaded = false;
    if (pageable) {
      ctx->atlas_recorded = &atlas_recorded;
      try { uploader = std::thread(upload); threaded = true; } catch (...) { ctx->atlas_recorded = nullptr; }   // no thread: upload inline
    }
    if (!threaded) upload();
  }
  SC_CUDA(cudaMemsetAsync(d_lab, 0, nvox, st));
  if (d_proba) SC_CUDA(cudaMemsetAsync(d_proba, 0, nvox * 60, st));
  const int seg_status = segment_volume(ctx, d_vol, dims, d_atlas, box, cand_mask_host ? d_mask : nullptr, d_lab, d_proba, st);
  if (uploader.joinable()) uploader.join();
  ctx->atlas_recorded = nullptr;
  if (ctx->atlas_ready) cudaStreamWaitEvent(st, ctx->atlas_ready, 0);  // join the side stream (the last chunk may not have been waited for)
  ctx->atlas_ready = nullptr;
  ctx->atlas_chunks = 0;
  SC_CHECK(upload_err.load() == 0, SC_ERR_CUDA, "sc_segment_volume_host: atlas upload failed: %s", cudaGetErrorString((cudaError_t)upload_err.load()));
  SC_TRY(seg_status);
  if (label_vol_host) SC_CUDA(cudaMemcpyAsync(label_vol_host, d_lab, nvox, cudaMemcpyDeviceToHost, st));
  if (proba_vol_host) SC_CUDA(cudaMemcpyAsync(proba_vol_host, d_proba, nvox * 60, cudaMemcpyDeviceToHost, st));
  SC_CUDA(cudaStreamSynchronize(st));
  joiner.ok = true;
  return SC_OK;
}

int sc_dense_layer(sc_ctx* ctx, int which, const float* in_dev, int64_t n, float* out_dev, int backend, void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_dense_layer", (cudaStream_t)stream));
  SC_CHECK(which >= 0 && which <= 4 && in_dev && out_dev && n > 0 && n < (1ll << 31), SC_ERR_ARG, "sc_dense_layer: bad argument");
  SC_CHECK(backend == 0 || (backend == 1 && ctx->tc_state), SC_ERR_UNSUPPORTED, "sc_dense_layer: back-end %d unavailable", backend);
  GemmProblem p;
  const GemmW* w;
  if (which < 3) {
    w = &ctx->br[which].d1;
    gemm_problem_rows(p, in_dev, kFeatLd, kFeatLd, (int)n);
    p.C = out_dev; p.ldc = 192; p.n_store = 192; p.prof_cls = PC_GEMM_D1;
  } else if (which == 3) {
    w = &ctx->fc1;
    gemm_problem_rows(p, in_dev, kFeatLd, kFeatLd, (int)n);
    p.C = out_dev; p.ldc = kH1Ld; p.n_store = 540; p.prof_cls = PC_GEMM_FC1;
  } else {
    w = &ctx->fc2;
    gemm_problem_rows(p, in_dev, kH1Ld, kH1Ld, (int)n);
    p.C = out_dev; p.ldc = kH2Ld; p.n_store = kH2Ld; p.prof_cls = PC_GEMM_FC2;
  }
  if (backend == 1) {  // the tcgen05 back-end consumes split bf16 hi|lo rows
    SC_TRY(ensure_ws(ctx->ws, (size_t)n * kFeatLd * sizeof(float)));
    float* tmp = reinterpret_cast<float*>(ctx->ws.ptr);
    SC_TRY(launch_split_rows(ctx, in_dev, n, tmp, (cudaStream_t)stream));
    p.A = p.a_base = tmp;
    return launch_gemm_tc(ctx, p, *w, (cudaStream_t)stream);
  }
  return launch_gemm(ctx, p, *w, (cudaStream_t)stream);
}

int sc_scatter(sc_ctx* ctx, const int32_t* xyz_dev, int64_t n, const int32_t* label_dev, const float* proba_dev,
               const int32_t dims[3], uint8_t* label_vol_dev, float* proba_vol_dev, void* stream) {
  SC_CHECK(ctx && (xyz_dev || n == 0) && n >= 0, SC_ERR_ARG, "sc_scatter: bad argument");
  SC_TRY(check_dims(dims, "sc_scatter"));
  SC_CUDA(cudaSetDevice(ctx->device));
  return launch_scatter(ctx, xyz_dev, n, label_dev, proba_dev, dims, label_vol_dev, proba_vol_dev, (cudaStream_t)stream);
}

int sc_train_forward_backward(sc_ctx* ctx, const float* in1_dev, const float* in2_dev, const float* in3_dev,
                              const float* in4_dev, const uint8_t* y_dev, int64_t n, int64_t n_global, uint64_t seed,
                              const uint8_t* drop_masks_dev, float* loss_dev, void* stream) {
  SC_TRY(need_weights(ctx, "sc_train_forward_backward"));
  SC_CHECK(n > 0 && n_global >= n, SC_ERR_ARG, "sc_train_forward_backward: bad batch size");
  SC_CHECK(in1_dev && in2_dev && in3_dev && in4_dev && y_dev && loss_dev, SC_ERR_ARG, "sc_train_forward_backward: null argument");
  return train_forward_backward(ctx, in1_dev, in2_dev, in3_dev, in4_dev, y_dev, n, n_global, seed, drop_masks_dev,
                                loss_dev, (cudaStream_t)stream);
}

int sc_grad_buffer(sc_ctx* ctx, float** grads_dev) {
  SC_CHECK(ctx && grads_dev, SC_ERR_ARG, "sc_grad_buffer: null argument");
  *grads_dev = ctx->grads;
  return SC_OK;
}

int sc_param_buffer(sc_ctx* ctx, float** params_dev) {
  SC_CHECK(ctx && params_dev, SC_ERR_ARG, "sc_param_buffer: null argument");
  *params_dev = ctx->params;
  return SC_OK;
}

int sc_adam_step(sc_ctx* ctx, float lr, float beta1, float beta2, float eps, float grad_scale, float stat_scale, void* stream) {
  SC_TRY(need_weights(ctx, "sc_adam_step"));
  return adam_step(ctx, lr, beta1, beta2, eps, grad_scale, stat_scale, (cudaStream_t)stream);
}

int sc_set_allreduce_hook(sc_ctx* ctx, sc_allreduce_fn fn, void* user) {
  SC_CHECK(ctx, SC_ERR_ARG, "sc_set_allreduce_hook: null context");
  ctx->ar_hook = fn; ctx->ar_user = user;
  return SC_OK;
}

int sc_fused_export(sc_ctx* ctx, unsigned char* handles_out) {
  SC_CHECK(ctx && handles_out, SC_ERR_ARG, "sc_fused_export: null argument");
  return fused_export(ctx, handles_out);
}
int sc_fused_attach(sc_ctx* ctx, int rank, int world, const unsigned char* all_handles) {
  SC_CHECK(ctx && all_handles, SC_ERR_ARG, "sc_fused_attach: null argument");
  return fused_attach(ctx, rank, world, all_handles);
}
int sc_allreduce_adam_step(sc_ctx* ctx, float lr, float beta1, float beta2, float eps, void* stream) {
  SC_TRY(need_weights(ctx, "sc_allreduce_adam_step"));
  return fused_allreduce_adam(ctx, lr, beta1, beta2, eps, (cudaStream_t)stream);
}

int sc_reset_optimizer(sc_ctx* ctx) {
  SC_CHECK(ctx, SC_ERR_ARG, "sc_reset_optimizer: null context");
  SC_CUDA(cudaSetDevice(ctx->device));
  SC_CUDA(cudaDeviceSynchronize());
  SC_CUDA(cudaMemset(ctx->adam_m, 0, sizeof(float) * SC_PARAM_FLOATS));
  SC_CUDA(cudaMemset(ctx->adam_v, 0, sizeof(float) * SC_PARAM_FLOATS));
  ctx->adam_t = 0;
  return SC_OK;
}

int sc_eval_batch(sc_ctx* ctx, const float* in1_dev, const float* in2_dev, const float* in3_dev, const float* in4_dev,
                  const uint8_t* y_dev, int64_t n, float* out2_dev, void* stream) {
  SC_TRY(fresh_weights(ctx, "sc_eval_batch", (cudaStream_t)stream));
  SC_CHECK(n > 0 && in1_dev && in2_dev && in3_dev && in4_dev && y_dev && out2_dev, SC_ERR_ARG, "sc_eval_batch: bad argument");
  return eval_batch(ctx, in1_dev, in2_dev, in3_dev, in4_dev, y_dev, n, out2_dev, (cudaStream_t)stream);
}

}  // extern "C"
