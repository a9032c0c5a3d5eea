// Monte-Carlo dropout over the FC head of the dense path (Gal & Ghahramani 2016).
//
// The network was trained with dropout p = 0.5 at three sites, each the INPUT of a dense layer: *_l1drop before each
// branch's d1, f1_drop before FC1 and f2_drop before fc_2 (its FC1 half; the atlas columns have none).  Pass t uses ONE
// keep mask for every voxel, keep[t][j] = hash3(seed, t * 2700 + j) & 1 in the training step's layout
// ([3][540] l1drop (k = c*9 + h*3 + w) | [540] f1_drop | [540] f2_drop), so a pass is the deterministic head with the
// weight rows of the dropped inputs zeroed and the kept ones doubled: W' = diag(2 keep) W.  Doubling is exact in bf16,
// so the masked split weights are the prepared hi / lo halves doubled or zeroed, with no rounding.  The convolutions
// (phase 1 of segment_volume) do not depend on the mask and run once; per slab, d1 x3, FC1 and fc_2 run once per pass
// with the masked copy, and fc_2's epilogue accumulates the softmax and sum_c p ln p of every row (gemm_tc.cu, MC_ACC).
// The finalize kernel turns the sums into the predictive mean, its entropy and the mutual information.
#include "common.cuh"

namespace sc {

constexpr int kMcD1Floats = 192 * kD1K;              // d1_dense of one branch: [Npad 192][Kpad 576]
constexpr int kMcFc1Floats = 576 * kFeatLd;          // FC1: [576][576]
constexpr int kMcFc2Floats = kH2Ld * kH1Ld;          // fc_2: [272][576]
constexpr int kMcFloats = 3 * kMcD1Floats + kMcFc1Floats + kMcFc2Floats;   // 820224 floats = 3.3 MB

struct McSrc { const uint32_t* w[5]; };               // the prepared w_nk of d1_dense x3, FC1, fc_2

// dropout unit j of logical K index k of matrix `mat` (0..2 d1 of a branch, 3 FC1, 4 fc_2), or -1 where no dropout applies
// (zero padding, fc_2's atlas rows)
__device__ __forceinline__ int mc_unit(int mat, int k) {
  if (mat < 3) {                                     // k = tap * 64 + c  <->  the flattened conv5 unit c * 9 + tap
    const int tap = k >> 6, c = k & 63;
    return c < 60 ? mat * 540 + c * 9 + tap : -1;
  }
  if (mat == 3) {                                    // feature row: 192 columns per view, 180 used
    const int view = k / 192, i = k - view * 192;
    return i < 180 ? 1620 + view * 180 + i : -1;
  }
  return k < 540 ? 2160 + k : -1;
}

// one 32-bit slot = two bf16 of one half (hi or lo) of a split row: logical k and k + 1
__global__ void __launch_bounds__(256) mc_mask_kernel(const McSrc src, uint32_t* __restrict__ dst, uint64_t seed, int t) {
  const int f = blockIdx.x * 256 + threadIdx.x;
  if (f >= kMcFloats) return;
  int mat, off;
  if (f < 3 * kMcD1Floats) { mat = f / kMcD1Floats; off = f - mat * kMcD1Floats; }
  else if (f < 3 * kMcD1Floats + kMcFc1Floats) { mat = 3; off = f - 3 * kMcD1Floats; }
  else { mat = 4; off = f - 3 * kMcD1Floats - kMcFc1Floats; }
  const int e = (off % kFeatLd) * 2;                 // bf16 index inside the row: per 64-wide k block 64 hi | 64 lo
  const int k = (e >> 7) * 64 + (e & 63);
  // a select chain rather than src.w[mat]: a run-time index would copy the parameter array to local memory
  const uint32_t* row = mat == 0 ? src.w[0] : mat == 1 ? src.w[1] : mat == 2 ? src.w[2] : mat == 3 ? src.w[3] : src.w[4];
  uint32_t v = __ldg(row + off);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int j = mc_unit(mat, k + i);
    if (j < 0) continue;
    const uint32_t sh = 16 * i;
    const uint32_t keep = hash3(seed, (uint64_t)t * kDropUnits + j) & 1u;
    const float w = __bfloat162float(__ushort_as_bfloat16((unsigned short)(v >> sh)));
    const uint32_t r = keep ? (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(2.f * w)) : 0u;   // exact: a power-of-two scale
    v = (v & ~(0xFFFFu << sh)) | (r << sh);
  }
  dst[f] = v;
}

int mc_prepare(sc_ctx* ctx, McWeights& w) {
  if (!ctx->mc_w) SC_CUDA(cudaMalloc(&ctx->mc_w, (size_t)kMcFloats * sizeof(float)));
  for (int b = 0; b < 3; ++b) { w.d1[b] = ctx->br[b].d1_dense; w.d1[b].w_nk = ctx->mc_w + b * kMcD1Floats; }
  w.fc1 = ctx->fc1; w.fc1.w_nk = ctx->mc_w + 3 * kMcD1Floats;
  w.fc2 = ctx->fc2; w.fc2.w_nk = ctx->mc_w + 3 * kMcD1Floats + kMcFc1Floats;
  SC_CHECK(w.d1[0].Npad * w.d1[0].Kpad == kMcD1Floats && w.fc1.Npad * w.fc1.Kpad == kMcFc1Floats &&
           w.fc2.Npad * w.fc2.Kpad == kMcFc2Floats, SC_ERR_STATE, "mc_prepare: unexpected weight layout");
  return SC_OK;
}

int launch_mc_mask(sc_ctx* ctx, uint64_t seed, int t, cudaStream_t st) {
  McSrc src;
  for (int b = 0; b < 3; ++b) src.w[b] = reinterpret_cast<const uint32_t*>(ctx->br[b].d1_dense.w_nk);
  src.w[3] = reinterpret_cast<const uint32_t*>(ctx->fc1.w_nk);
  src.w[4] = reinterpret_cast<const uint32_t*>(ctx->fc2.w_nk);
  ProfScope prof(ctx, PC_MC, st);
  mc_mask_kernel<<<(kMcFloats + 255) / 256, 256, 0, st>>>(src, reinterpret_cast<uint32_t*>(ctx->mc_w), seed, t);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// row m of the slab accumulator: {sum_t p_t[0..14], sum_t sum_c p_t,c ln p_t,c} -> label / mean / entropy / mutual information
// of its voxel, with fc_2's row -> voxel mapping (compacted rows through rowvox, the box geometry, the candidate mask)
__global__ void __launch_bounds__(256) mc_finalize_kernel(const float* __restrict__ acc, int64_t rows, int samples,
                                                          const int32_t* __restrict__ rowvox, OutGeo g, const uint8_t* __restrict__ mask,
                                                          uint8_t* __restrict__ label, float* __restrict__ proba,
                                                          float* __restrict__ entropy, float* __restrict__ mi) {
  const int64_t m = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (m >= rows) return;
  const int64_t r = rowvox ? (int64_t)__ldg(rowvox + m) : m;
  const int64_t plane = (int64_t)g.by * g.bz;
  const int ix = (int)(r / plane);
  const int rem = (int)(r - (int64_t)ix * plane);
  const int iy = rem / g.bz, iz = rem - iy * g.bz;
  const int64_t o = ((int64_t)(g.x0 + ix) * g.Y + (g.y0 + iy)) * g.Z + (g.z0 + iz);
  if (mask && mask[o] == 0) return;
  const float4* a4 = reinterpret_cast<const float4*>(acc + m * 16);
  float s[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 v = __ldg(a4 + i);
    s[4 * i] = v.x; s[4 * i + 1] = v.y; s[4 * i + 2] = v.z; s[4 * i + 3] = v.w;
  }
  const float T = (float)samples;
  float p[15];
  int best = 0;
  float bp = s[0] / T;
#pragma unroll
  for (int c = 0; c < 15; ++c) {
    p[c] = s[c] / T;
    if (p[c] > bp) { bp = p[c]; best = c; }      // first maximum wins (np.argmax)
  }
  const float H = -plogp15(p);
  if (label) label[o] = (uint8_t)best;
  if (proba) {
#pragma unroll
    for (int c = 0; c < 15; ++c) proba[o * 15 + c] = p[c];
  }
  if (entropy) entropy[o] = H;
  if (mi) mi[o] = fmaxf(0.f, H + s[15] / T);      // H(mean) - mean of H(p_t); exactly 0 for one pass
}

int launch_mc_finalize(sc_ctx* ctx, const float* acc, int64_t rows, int samples, const int32_t* rowvox, const OutGeo& geo,
                       const uint8_t* mask, uint8_t* label, float* proba, float* entropy, float* mi, cudaStream_t st) {
  if (rows <= 0) return SC_OK;
  ProfScope prof(ctx, PC_MC, st);
  mc_finalize_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(acc, rows, samples, rowvox, geo, mask, label, proba, entropy, mi);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
