// Fine-tuning the pretrained network on a new domain (Kushibar et al., Sci. Rep. 2019): the convolutional trunk (conv1..conv5
// with BatchNorm and PReLU, all three views) is frozen and evaluated in deterministic mode, so the conv5 features of a sample
// never change.  They are computed once per training sample (trunk_features) and kept on the device as float32 rows
// [N][3][540], k = c*9 + h*3 + w per view: the input of <view>_d1 before dropout.  The head (d1 x3, FC1, fc_2, out_layer and
// their PReLUs) then trains from those rows:
//   - the training step (train.cu: head_train_forward_backward) is train_body from d1 on, fed by head_gather_kernel;
//   - the validation pass (head_eval_batch) is the deterministic inference head on the same rows;
//   - freeze_trunk marks the trunk entries of the optimiser's `trainable` map 2, which both Adam kernels leave untouched.
#include "common.cuh"

namespace sc {

// ---- trunk features ----------------------------------------------------------------------------------------------------
// conv5 map of one view (branch_trunk_tc: [7][n][8] pixels of 64 bf16 hi | 64 bf16 lo channel slots, BatchNorm and PReLU
// applied, valid 3x3 region) -> out[i * 1620 + k] = hi + lo of channel c at (h, w), k = c*9 + h*3 + w
__global__ void c5_features_kernel(const float* __restrict__ c5, int n, float* __restrict__ out /* + view * 540 */) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)n * 540) return;
  const int i = (int)(e / 540), k = (int)(e - (int64_t)i * 540);
  const int c = k / 9, r = k - c * 9, h = r / 3, w = r - h * 3;
  const __nv_bfloat16* px = reinterpret_cast<const __nv_bfloat16*>(c5) + ((int64_t)h * n * 8 + (int64_t)i * 8 + w) * 128;
  out[(int64_t)i * kTrunkFeat + k] = __bfloat162float(px[c]) + __bfloat162float(px[64 + c]);
}

// the tensor-core patchwise trunk of forward_patches, 4096 patches per pass
int trunk_features(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, int64_t n, float* feats, cudaStream_t st) {
  const int64_t sub = 4096;
  const int64_t cmax = n < sub ? n : sub;
  SC_TRY(ensure_ws(ctx->ws, branch_patches_tc_bytes(cmax)));
  float* scratch = reinterpret_cast<float*>(ctx->ws.ptr);
  const float* ins[3] = {in1, in2, in3};
  for (int64_t s = 0; s < n; s += sub) {
    const int64_t m = n - s < sub ? n - s : sub;
    for (int b = 0; b < 3; ++b) {
      float* c5 = nullptr;
      SC_TRY(branch_trunk_tc(ctx, b, ins[b] + s * 1024, m, scratch, &c5, st));
      ProfScope prof(ctx, PC_HEAD, st);
      c5_features_kernel<<<(unsigned)((m * 540 + 255) / 256), 256, 0, st>>>(c5, (int)m, feats + s * kTrunkFeat + b * 540);
      ctx->launches++;
      SC_CUDA(cudaGetLastError());
    }
  }
  return SC_OK;
}

// ---- d1's operands from the feature table --------------------------------------------------------------------------------
// One CTA per tile of 64 batch entries x 64 feature columns of one view (grid: entry tiles x 9 column blocks x 3 views).  The
// tile is read with the columns fastest (256 B runs of a feature row), dropout-masked (x2 / x0) in shared memory, and written
// as 64-entry blocks of both split layouts d1 consumes: row-major F5s [n][576] (columns 540..575 as zeros, the K padding) and,
// when asked for, transposed F5T [576][npad] (the wgrad operand).  The CTAs of view 0, column block 0 also gather the atlas rows
// and labels of their entries.  Row indices are trusted (the caller range-checks them, as for sc_gather_samples).
__global__ void __launch_bounds__(256) head_gather_kernel(const HeadGather g) {
  __shared__ float tile[64][65];
  __shared__ int64_t rows[64];
  const int m0 = blockIdx.x * 64, kb = blockIdx.y, b = blockIdx.z, k0 = kb * 64;
  const int tid = threadIdx.x;
  float* const f5s = b == 0 ? g.F5s[0] : b == 1 ? g.F5s[1] : g.F5s[2];   // (a dynamic index into the parameter arrays costs a stack copy)
  float* const f5t = b == 0 ? g.F5T[0] : b == 1 ? g.F5T[1] : g.F5T[2];
  if (tid < 64) {
    const int m = m0 + tid;
    rows[tid] = m < g.n ? (g.idx ? g.idx[m] : g.row0 + m) : -1;
  }
  __syncthreads();
  for (int e = tid; e < 64 * 64; e += 256) {
    const int r = e >> 6, c = e & 63, k = k0 + c;
    float v = 0.f;
    if (rows[r] >= 0 && k < 540) {
      v = __ldg(g.feats + rows[r] * kTrunkFeat + b * 540 + k);
      if (g.masks) v = g.masks[(int64_t)(m0 + r) * kDropUnits + b * 540 + k] ? 2.f * v : 0.f;
    }
    tile[r][c] = v;
  }
  __syncthreads();
  for (int e = tid; e < 64 * 64; e += 256) {   // row-major: column fastest
    const int r = e >> 6, c = e & 63;
    if (rows[r] >= 0) store_row1(f5s + (int64_t)(m0 + r) * 576, k0 + c, 1, tile[r][c]);
  }
  if (f5t) {
    for (int e = tid; e < 64 * 64; e += 256) {   // transposed: entry fastest
      const int c = e >> 6, r = e & 63;
      if (rows[r] >= 0 && k0 + c < 540) store_row1(f5t + (int64_t)(k0 + c) * g.npad, m0 + r, 1, tile[r][c]);
    }
  }
  if (kb == 0 && b == 0) {
    for (int e = tid; e < 64 * 15; e += 256) {
      const int r = e / 15, j = e - r * 15;
      if (rows[r] >= 0) g.in4[(int64_t)(m0 + r) * 15 + j] = __ldg(g.atlas_rows + rows[r] * 15 + j);
    }
    if (tid < 64 && rows[tid] >= 0) g.y[m0 + tid] = g.labels[rows[tid]];
  }
}

int launch_head_gather(sc_ctx* ctx, const HeadGather& g, cudaStream_t st) {
  ProfScope prof(ctx, PC_HEAD, st);
  head_gather_kernel<<<dim3((unsigned)((g.n + 63) / 64), 9, 3), 256, 0, st>>>(g);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---- validation on the feature table -------------------------------------------------------------------------------------
// deterministic head on rows idx[0..n) (sc_eval_batch's outputs), in chunks of 32768 rows: gather -> d1 x3 (the patchwise
// inference weights, K = 540 in (c, h, w) order) -> FC1 -> atlas -> fc_2 + out_layer / softmax -> loss and correct count
int head_eval_batch(sc_ctx* ctx, const float* feats, const float* atlas_rows, const uint8_t* labels, const int64_t* idx, int64_t n,
                    float* out2, cudaStream_t st) {
  const int64_t chunk = 32768;
  const int64_t cmax = n < chunk ? n : chunk;
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t rows_b = al((size_t)cmax * 576 * 4);
  SC_TRY(ensure_ws(ctx->ws, 5 * rows_b + al((size_t)cmax * 15 * 4) * 2 + al((size_t)cmax)));
  char* p = reinterpret_cast<char*>(ctx->ws.ptr);
  float* x[3];
  for (int b = 0; b < 3; ++b) { x[b] = reinterpret_cast<float*>(p); p += rows_b; }
  float* d1 = reinterpret_cast<float*>(p); p += rows_b;
  float* h1 = reinterpret_cast<float*>(p); p += rows_b;
  float* in4 = reinterpret_cast<float*>(p); p += al((size_t)cmax * 15 * 4);
  float* proba = reinterpret_cast<float*>(p); p += al((size_t)cmax * 15 * 4);
  uint8_t* y = reinterpret_cast<uint8_t*>(p);
  SC_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(float), st));
  for (int64_t s = 0; s < n; s += chunk) {
    const int64_t m = n - s < chunk ? n - s : chunk;
    HeadGather g;
    g.feats = feats; g.atlas_rows = atlas_rows; g.labels = labels;
    g.idx = idx ? idx + s : nullptr; g.row0 = s; g.n = (int)m; g.masks = nullptr;
    for (int b = 0; b < 3; ++b) { g.F5s[b] = x[b]; g.F5T[b] = nullptr; }
    g.npad = 0; g.in4 = in4; g.y = y;
    SC_TRY(launch_head_gather(ctx, g, st));
    for (int b = 0; b < 3; ++b) {
      GemmProblem q;
      gemm_problem_rows(q, x[b], kFeatLd, kFeatLd, (int)m);
      q.C = d1; q.ldc = kFeatLd; q.c_col0 = b * 192; q.n_store = 192; q.out_split = 1; q.prof_cls = PC_GEMM_D1;
      SC_TRY(launch_gemm_tc(ctx, q, ctx->br[b].d1, st));
    }
    SC_TRY(head_rows(ctx, d1, in4, m, h1, nullptr, proba, nullptr, st));
    SC_TRY(launch_eval_reduce(ctx, proba, y, m, out2, st));
  }
  return SC_OK;
}

// ---- the optimiser's map ---------------------------------------------------------------------------------------------------
// 1: Adam; 0: BatchNorm running mean / inv_std (s <- 0.9 s + 0.1 slot); 2 (frozen trunk): untouched.  The trunk of a view is
// the contiguous run of its conv1..conv5 arrays (W, BN beta / gamma / mean / inv_std, PReLU alpha) in the parameter layout.
int freeze_trunk(sc_ctx* ctx, bool frozen) {
  std::vector<uint8_t> t(SC_PARAM_FLOATS, 1);
  for (int b = 0; b < 3; ++b) {
    const BranchOff& O = ctx->off.br[b];
    for (int l = 0; l < 5; ++l)
      for (int k = 2; k < 4; ++k)
        for (int c = 0; c < kConvCout[l]; ++c) t[O.bn[l][k] + c] = 0;
    if (frozen)
      for (int i = O.convW[0]; i < O.d1W; ++i) t[i] = 2;
  }
  SC_CUDA(cudaMemcpy(ctx->trainable, t.data(), SC_PARAM_FLOATS, cudaMemcpyHostToDevice));
  ctx->trunk_frozen = frozen;
  return SC_OK;
}

}  // namespace sc
