// Patchwise forward: net.predict_proba on {'in1','in2','in3','in4'} (call sites
// cnn_cort/base.py:425-438; graph cnn_cort/nets.py:170-231), deterministic mode.
//
// branch_patch_kernel: one CTA per (patch, view) keeps conv1..conv5 of that patch in shared
// memory (conv -> BN affine -> PReLU, 2x2 max-pools after conv2 and conv4, in that order:
// trained PReLU slopes are negative or > 1, so pooling cannot move before the activation)
// and emits the flattened 60x3x3 map (k = c*9 + h*3 + w).  d1 / FC1 / fc_2 then run as
// GEMMs over the whole batch (gemm_simt.cu or gemm_tc.cu), out_layer+softmax last (on the tensor cores: in
// fc_2's epilogue).
#include "common.cuh"

namespace sc {

struct PatchW {
  const float* c1_w;
  const float* w[5];
  const float* scale[5];
  const float* shift[5];
  const float* alpha[5];
};

constexpr int C1_LD = 32;                 // conv1 map rows padded 30 -> 32
constexpr int S_IN = 0;                   // 1024
constexpr int S_C1 = 1024;                // 20*30*32 = 19200  (conv3 output overlays it later)
constexpr int S_P1 = S_C1 + 19200;        // 20*14*16 = 4480
constexpr int S_P2 = S_P1 + 4480;         // 40*25 = 1000
constexpr int S_TOTAL = S_P2 + 1000;
constexpr size_t PATCH_SMEM = S_TOTAL * sizeof(float);

__global__ void __launch_bounds__(256) branch_patch_kernel(const float* __restrict__ patches, const PatchW W,
                                                           float* __restrict__ c5_out, int round_out) {
  extern __shared__ __align__(16) float sm[];
  float* s_in = sm + S_IN;
  float* s_c1 = sm + S_C1;
  float* s_c3 = sm + S_C1;  // overlay: conv1 map is dead once pool1 exists
  float* s_p1 = sm + S_P1;
  float* s_p2 = sm + S_P2;
  const int tid = threadIdx.x;
  const int64_t n = blockIdx.x;
  reinterpret_cast<float4*>(s_in)[tid] = __ldg(reinterpret_cast<const float4*>(patches + n * 1024) + tid);
  __syncthreads();

  // conv1: 1 -> 20, 30x30
  for (int idx = tid; idx < 900; idx += 256) {
    const int py = idx / 30, px = idx - py * 30;
    float x[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) x[ky * 3 + kx] = s_in[(py + ky) * 32 + px + kx];
#pragma unroll 5
    for (int co = 0; co < 20; ++co) {
      float a = 0.f;
#pragma unroll
      for (int t = 0; t < 9; ++t) a = fmaf(x[t], __ldg(W.c1_w + t * 20 + co), a);
      s_c1[(co * 30 + py) * C1_LD + px] = prelu(fmaf(a, __ldg(W.scale[0] + co), __ldg(W.shift[0] + co)), __ldg(W.alpha[0] + co));
    }
  }
  __syncthreads();

  // conv2 (20 -> 20, 28x28) + pool -> 14x14.  item = 4 channels x one pooled pixel (2x2 conv outputs)
  for (int item = tid; item < 5 * 196; item += 256) {
    const int cgp = item / 196, pp = item - cgp * 196, ppy = pp / 14, ppx = pp - ppy * 14;
    float acc[4][4];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[p][c] = 0.f;
#pragma unroll 2
    for (int ci = 0; ci < 20; ++ci) {
      float x[4][4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float2* src = reinterpret_cast<const float2*>(s_c1 + (ci * 30 + 2 * ppy + r) * C1_LD + 2 * ppx);
        const float2 a = src[0], b = src[1];
        x[r][0] = a.x; x[r][1] = a.y; x[r][2] = b.x; x[r][3] = b.y;
      }
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(W.w[1] + (ci * 9 + ky * 3 + kx) * 20 + cgp * 4));
          const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
          for (int dy = 0; dy < 2; ++dy)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx)
#pragma unroll
              for (int c = 0; c < 4; ++c) acc[dy * 2 + dx][c] = fmaf(x[dy + ky][dx + kx], wv[c], acc[dy * 2 + dx][c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int co = cgp * 4 + c;
      const float s = __ldg(W.scale[1] + co), h = __ldg(W.shift[1] + co), al = __ldg(W.alpha[1] + co);
      float m = prelu(fmaf(acc[0][c], s, h), al);
#pragma unroll
      for (int p = 1; p < 4; ++p) m = fmaxf(m, prelu(fmaf(acc[p][c], s, h), al));
      s_p1[(co * 14 + ppy) * 16 + ppx] = m;
    }
  }
  __syncthreads();

  // conv3 (20 -> 40, 12x12).  item = 8 channels x 4 consecutive pixels of a row
  if (tid < 5 * 36) {
    const int cgp = tid / 36, seg = tid - cgp * 36, row = seg / 3, c0 = (seg - row * 3) * 4;
    float acc[4][8];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[p][c] = 0.f;
#pragma unroll 1
    for (int ci = 0; ci < 20; ++ci) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const float* src = s_p1 + (ci * 14 + row + ky) * 16 + c0;
        const float4 a = *reinterpret_cast<const float4*>(src);
        const float2 b = *reinterpret_cast<const float2*>(src + 4);
        const float x[6] = {a.x, a.y, a.z, a.w, b.x, b.y};
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float4* wp = reinterpret_cast<const float4*>(W.w[2] + (ci * 9 + ky * 3 + kx) * 40 + cgp * 8);
          const float4 w0 = __ldg(wp), w1 = __ldg(wp + 1);
          const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
          for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[p][c] = fmaf(x[p + kx], wv[c], acc[p][c]);
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int co = cgp * 8 + c;
      const float s = __ldg(W.scale[2] + co), h = __ldg(W.shift[2] + co), al = __ldg(W.alpha[2] + co);
#pragma unroll
      for (int p = 0; p < 4; ++p) s_c3[(co * 12 + row) * 12 + c0 + p] = prelu(fmaf(acc[p][c], s, h), al);
    }
  }
  __syncthreads();

  // conv4 (40 -> 40, 10x10) + pool -> 5x5.  item = 4 channels x one pooled pixel
  if (tid < 250) {
    const int cgp = tid / 25, pp = tid - cgp * 25, ppy = pp / 5, ppx = pp - ppy * 5;
    float acc[4][4];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[p][c] = 0.f;
#pragma unroll 2
    for (int ci = 0; ci < 40; ++ci) {
      float x[4][4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float2* src = reinterpret_cast<const float2*>(s_c3 + (ci * 12 + 2 * ppy + r) * 12 + 2 * ppx);
        const float2 a = src[0], b = src[1];
        x[r][0] = a.x; x[r][1] = a.y; x[r][2] = b.x; x[r][3] = b.y;
      }
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(W.w[3] + (ci * 9 + ky * 3 + kx) * 40 + cgp * 4));
          const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
          for (int dy = 0; dy < 2; ++dy)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx)
#pragma unroll
              for (int c = 0; c < 4; ++c) acc[dy * 2 + dx][c] = fmaf(x[dy + ky][dx + kx], wv[c], acc[dy * 2 + dx][c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int co = cgp * 4 + c;
      const float s = __ldg(W.scale[3] + co), h = __ldg(W.shift[3] + co), al = __ldg(W.alpha[3] + co);
      float m = prelu(fmaf(acc[0][c], s, h), al);
#pragma unroll
      for (int p = 1; p < 4; ++p) m = fmaxf(m, prelu(fmaf(acc[p][c], s, h), al));
      s_p2[co * 25 + pp] = m;
    }
  }
  __syncthreads();

  // conv5 (40 -> 60, 3x3) -> global, flattened (c, h, w)
  float* out = c5_out + n * kFeatLd;
  if (tid < 135) {
    const int cgp = tid / 9, px = tid - cgp * 9, py = px / 3, pxx = px - py * 3;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int ci = 0; ci < 40; ++ci) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float x = s_p2[ci * 25 + (py + ky) * 5 + pxx + kx];
          const float4 w = __ldg(reinterpret_cast<const float4*>(W.w[4] + (ci * 9 + ky * 3 + kx) * 60 + cgp * 4));
          acc[0] = fmaf(x, w.x, acc[0]); acc[1] = fmaf(x, w.y, acc[1]);
          acc[2] = fmaf(x, w.z, acc[2]); acc[3] = fmaf(x, w.w, acc[3]);
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int co = cgp * 4 + c;
      const float v = prelu(fmaf(acc[c], __ldg(W.scale[4] + co), __ldg(W.shift[4] + co)), __ldg(W.alpha[4] + co));
      store_row1(out, co * 9 + px, round_out, v);
    }
  } else if (tid >= 220) {
    store_row1(out, 540 + (tid - 220), round_out, 0.f);   // K padding 540..575
  }
}

int launch_branch_patches(sc_ctx* ctx, int b, const float* patches, int64_t n, float* c5_out, cudaStream_t st) {
  if (n == 0) return SC_OK;
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(branch_patch_kernel), (int)PATCH_SMEM));
  PatchW W;
  W.c1_w = ctx->br[b].c1_w;
  for (int l = 0; l < 5; ++l) {
    W.w[l] = ctx->br[b].conv_w[l];
    W.scale[l] = ctx->br[b].scale[l]; W.shift[l] = ctx->br[b].shift[l]; W.alpha[l] = ctx->br[b].alpha[l];
  }
  SC_CHECK(n < (1ll << 31), SC_ERR_ARG, "forward: batch too large");
  ProfScope prof(ctx, PC_PATCH_BRANCH, st);
  branch_patch_kernel<<<(unsigned)n, 256, PATCH_SMEM, st>>>(patches, W, c5_out, ctx->gemm_backend == 1);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// [n][15] atlas rows -> columns 540..575 of h1 (no background fix here: the caller's in4 already has it);
// also clears the K padding (columns 540..575) of the feature rows.
__global__ void atlas_rows_kernel(const float* __restrict__ in4, int64_t n, float* __restrict__ h1, int split) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 9) return;
  const int64_t m = i / 9;
  const int q = (int)(i - m * 9);
  float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (q * 4 + k < 15) a[k] = __ldg(in4 + m * 15 + q * 4 + k);
  store_row4(h1 + m * kH1Ld, 540 + 4 * q, split, a[0], a[1], a[2], a[3]);
}

int forward_patches(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, const float* in4, int64_t n,
                    float* proba, int32_t* label, cudaStream_t st) {
  const bool tc = ctx->gemm_backend == 1;
  const int64_t chunk = 32768, sub = 4096;      // head rows per pass / patches per tensor-core conv pass
  const size_t row_floats = 3 * kFeatLd + kFeatLd + kH1Ld + (tc ? 0 : kH2Ld);   // tensor-core mode: no h2 rows (fused into fc_2)
  const int64_t cmax = n < chunk ? n : chunk;
  const size_t head_bytes = (size_t)cmax * row_floats * sizeof(float) + 1024;
  const size_t conv_bytes = tc ? branch_patches_tc_bytes(cmax < sub ? cmax : sub) : 0;
  SC_TRY(ensure_ws(ctx->ws, head_bytes + conv_bytes));
  float* c5 = reinterpret_cast<float*>(ctx->ws.ptr);
  float* feats = c5 + (size_t)cmax * 3 * kFeatLd;
  float* h1 = feats + (size_t)cmax * kFeatLd;
  float* h2 = h1 + (size_t)cmax * kH1Ld;
  float* conv_scratch = reinterpret_cast<float*>(reinterpret_cast<char*>(ctx->ws.ptr) + ((head_bytes + 255) & ~(size_t)255));
  const float* ins[3] = {in1, in2, in3};
  for (int64_t s = 0; s < n; s += chunk) {
    const int64_t m = n - s < chunk ? n - s : chunk;
    for (int b = 0; b < 3; ++b) {
      if (tc) {   // conv1..conv5 + d1 on the tensor cores, 4096 patches at a time
        for (int64_t t = 0; t < m; t += sub) {
          const int64_t mm = m - t < sub ? m - t : sub;
          SC_TRY(branch_patches_tc(ctx, b, ins[b] + (s + t) * 1024, mm, conv_scratch, feats + t * kFeatLd, st));
        }
        continue;
      }
      float* c5b = c5 + (size_t)b * cmax * kFeatLd;
      SC_TRY(launch_branch_patches(ctx, b, ins[b] + s * 1024, m, c5b, st));
      GemmProblem p;
      gemm_problem_rows(p, c5b, kFeatLd, kFeatLd, (int)m);
      p.C = feats; p.ldc = kFeatLd; p.c_col0 = b * 192;
      p.n_store = 192; p.out_split = 0; p.prof_cls = PC_GEMM_D1;
      SC_TRY(launch_gemm(ctx, p, ctx->br[b].d1, st));
    }
    SC_TRY(head_rows(ctx, feats, in4 + s * 15, m, h1, h2, proba ? proba + s * 15 : nullptr, label ? label + s : nullptr, st));
  }
  return SC_OK;
}

int head_rows(sc_ctx* ctx, const float* feats, const float* in4, int64_t m, float* h1, float* h2, float* proba, int32_t* label,
              cudaStream_t st) {
  const bool tc = ctx->gemm_backend == 1;
  GemmProblem p;
  gemm_problem_rows(p, feats, kFeatLd, kFeatLd, (int)m);
  p.C = h1; p.ldc = kH1Ld; p.n_store = 540; p.out_split = tc ? 1 : 0;
  p.prof_cls = PC_GEMM_FC1;
  SC_TRY(tc ? launch_gemm_tc(ctx, p, ctx->fc1, st) : launch_gemm(ctx, p, ctx->fc1, st));
  { ProfScope prof(ctx, PC_ATLAS, st);   // after FC1 (whose epilogue may zero columns 540..543)
    atlas_rows_kernel<<<(unsigned)((m * 9 + 255) / 256), 256, 0, st>>>(in4, m, h1, tc ? 1 : 0); }
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  gemm_problem_rows(p, h1, kH1Ld, kH1Ld, (int)m);
  p.n_store = kH2Ld; p.prof_cls = PC_GEMM_FC2;
  if (tc) {   // fc_2 with the out_layer and softmax / argmax in its epilogue
    SoftmaxOut smo = {proba, label, nullptr, nullptr, OutGeo{}, 0, nullptr};
    p.C = nullptr; p.ldc = 0; p.sm = &smo;
    return launch_gemm_tc(ctx, p, ctx->fc2, st);
  }
  p.C = h2; p.ldc = kH2Ld;
  SC_TRY(launch_gemm(ctx, p, ctx->fc2, st));
  return launch_out_softmax(ctx, h2, m, proba, label, nullptr, nullptr, nullptr, st);
}

}  // namespace sc
