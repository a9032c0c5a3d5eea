// Training step on the tensor cores (nolearn's train_fn inside net.fit, cnn_cort/nets.py:233-246).
//
// Same mathematics as train.cu (the exact-fp32 SIMT cross-check), different machinery:
//   * activations live in the wide-row split-bf16 maps of conv_sweep.cu (patches side by side, pixel = 32 or 64 channel
//     slots of bf16 hi | lo), so the convolutions run on the strip-sweep tcgen05 kernels:
//       forward  conv2..conv5   = the inference sweep with an identity epilogue (raw pre-BatchNorm output; the batch
//                                 statistics need a grid-wide reduction before the activation)
//       dgrad    conv2..conv5   = the same sweep over the zero-framed output gradient with the raw (un-flipped) taps and
//                                 the channel roles swapped
//       wgrad    conv2..conv5   = wgrad_mn_kernel below: an implicit GEMM whose K dimension is the PIXEL axis
//                                 (gW[tap][ci][co] = sum_p A[p + shift(tap)][ci] * dX[p][co]) with both operands MN-major, read
//                                 straight from the pixel-major maps (a TMA box of a map IS the canonical MN-major operand; a tap
//                                 is a shift of the outer TMA coordinate / a row-shifted descriptor start).  Its predecessor
//                                 wgrad_tc_kernel (sc_set_option "train_wgrad_mn" = 0) reads K-major operands from channel-major
//                                 ("planar transposed") bf16 hi/lo copies that the element-wise kernels then write next to the
//                                 pixel-major maps -- the gradient three times, shifted by 0, 1 and 2 pixels, because a filter
//                                 COLUMN would be a 2-byte shift of the innermost TMA coordinate, which must stay 16-byte aligned
//   * every product is the bf16x3 split (xl*wh + xh*wl + xh*wh, fp32 accumulate in TMEM), like inference
//   * BatchNorm statistics / activation / pooling and their backward passes are element-wise kernels over the split maps
// conv1 (K = 9) stays on CUDA cores.  The dense layers are in train_dense.cu.
#include "tc_common.cuh"

namespace sc {

__device__ __forceinline__ void tmem_ld16_raw(uint32_t taddr, uint32_t (&r)[16]) {   // 32 lanes x 16 consecutive 32-bit columns (no wait)
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

// ---------------------------------------------------------------------------------------------------------------
// split-map access: a pixel holds FMT channel slots as FMT bf16 "hi" then FMT bf16 "lo"; chunk = 8 channels = 16 B + 16 B
// ---------------------------------------------------------------------------------------------------------------
template <int FMT>
__device__ __forceinline__ void load8(const float* map, int64_t pixel, int chunk, float (&v)[8]) {
  const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(map) + pixel * (FMT * 4)) + chunk;
  const uint4 h = __ldg(p), l = __ldg(p + FMT / 8);
  const uint32_t hh[4] = {h.x, h.y, h.z, h.w}, ll[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    v[2 * k] = __uint_as_float(hh[k] << 16) + __uint_as_float(ll[k] << 16);
    v[2 * k + 1] = __uint_as_float(hh[k] & 0xffff0000u) + __uint_as_float(ll[k] & 0xffff0000u);
  }
}
__device__ __forceinline__ void split8(const float (&v)[8], uint4& h, uint4& l) {
  uint32_t hh[4], ll[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) split2(v[2 * k], v[2 * k + 1], hh[k], ll[k]);
  h = make_uint4(hh[0], hh[1], hh[2], hh[3]);
  l = make_uint4(ll[0], ll[1], ll[2], ll[3]);
}
template <int FMT>
__device__ __forceinline__ void store8(float* map, int64_t pixel, int chunk, const uint4& h, const uint4& l) {
  uint4* p = reinterpret_cast<uint4*>(reinterpret_cast<char*>(map) + pixel * (FMT * 4)) + chunk;
  p[0] = h;
  p[FMT / 8] = l;
}

// ---------------------------------------------------------------------------------------------------------------
// weight panels of the sweep kernels, re-derived from the master parameters on the device every step
// (same layout as weights.cu builds on the host for inference)
// ---------------------------------------------------------------------------------------------------------------
struct PanelJob { const float* W; int cout, cin, dgrad, ksteps, bn; uint16_t* plain; uint16_t* pair; };
struct PanelJobs { PanelJob j[8]; };
// one launch per branch: blockIdx.y = (layer 1..4) x (forward | dgrad)
__global__ void derive_panels_kernel(const PanelJobs jobs) {
  const PanelJob& J = jobs.j[blockIdx.y];
  const int cout = J.cout, cin = J.cin, dgrad = J.dgrad, ksteps = J.ksteps, bn = J.bn;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * cin * 9) return;
  const int t = i % 9, ci = (i / 9) % cin, co = i / (9 * cin);
  const float v = J.W[i];
  // forward: true convolution -> correlation taps (tap 8 - t), rows = output channels, k = input channels
  // dgrad:   raw taps, rows = the layer's INPUT channels, k = its output channels
  const int o = dgrad ? ci : co, k = dgrad ? co : ci, tap = dgrad ? t : 8 - t;
  const __nv_bfloat16 hb16 = __float2bfloat16_rn(v);
  const uint16_t hi = __bfloat16_as_ushort(hb16);
  const uint16_t lo = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(hb16)));
  size_t ip, iq;
  sweep_panel_pos(o, tap / 3, tap % 3, k, ksteps, bn, ip, iq);
  J.plain[ip] = hi;
  J.plain[ip + (size_t)3 * bn * 64] = lo;
  J.pair[iq] = hi;
  J.pair[iq + (size_t)3 * bn / 2 * 64] = lo;
}

// ---------------------------------------------------------------------------------------------------------------
// conv1 (1 -> 20, K = 9) from the staged patches into the F32CH map [30][n][32]; taps from device memory
// (graph-replayable), raw output (identity epilogue).  One thread per map position; columns 30, 31 are zero.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tconv1_kernel(const float* __restrict__ patches, int n, const float* __restrict__ wf /*[9][20]*/,
                                                     float* __restrict__ X0) {
  __shared__ float sw[180];
  for (int i = threadIdx.x; i < 180; i += 256) sw[i] = wf[i];
  __syncthreads();
  const int64_t total = (int64_t)30 * n * 32;
  for (int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x; p < total; p += (int64_t)gridDim.x * 256) {
    const int c = (int)(p & 31);
    const int s = (int)((p >> 5) % n);
    const int r = (int)(p / ((int64_t)n * 32));
    float v[24];
#pragma unroll
    for (int k = 0; k < 24; ++k) v[k] = 0.f;
    if (c < 30) {
      const float* src = patches + (int64_t)s * 1024 + r * 32 + c;
      float x[9];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) x[ky * 3 + kx] = __ldg(src + ky * 32 + kx);
#pragma unroll
      for (int co = 0; co < 20; ++co) {
        float a = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) a = fmaf(x[t], sw[t * 20 + co], a);
        v[co] = a;
      }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float w8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) w8[j] = v[8 * k + j];
      uint4 h, l;
      split8(w8, h, l);
      store8<32>(X0, p, k, h, l);
    }
    store8<32>(X0, p, 3, make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u));
  }
}

// ---------------------------------------------------------------------------------------------------------------
// BatchNorm batch statistics over the valid H x H region of a raw conv map (per channel sum and sum of squares)
// ---------------------------------------------------------------------------------------------------------------
template <int FMT>
__global__ void __launch_bounds__(256) tbn_stats_kernel(const float* __restrict__ X, int n, int C, int H, int Pw, int pitch,
                                                        double* __restrict__ sums /*[64][2]*/) {
  constexpr int NCH = FMT / 8;
  __shared__ float red[64][2];
  for (int i = threadIdx.x; i < 128; i += 256) (&red[0][0])[i] = 0.f;
  __syncthreads();
  const int chunk = threadIdx.x % NCH, slot = threadIdx.x / NCH;
  const int64_t total = (int64_t)H * n * H;
  float s[8], q[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = q[k] = 0.f;
  if (chunk * 8 < C) {
    const int64_t stride = (int64_t)gridDim.x * (256 / NCH);
    auto pos = [&](int64_t v) {
      const int c = (int)(v % H);
      const int sidx = (int)((v / H) % n);
      const int r = (int)(v / ((int64_t)H * n));
      return (int64_t)r * Pw + (int64_t)sidx * pitch + c;
    };
    // four points per iteration, all loads issued before the first is consumed (the grid stays small: every CTA ends with
    // same-address double atomics, which serialise at ~ 27 clk each)
    for (int64_t v = (int64_t)blockIdx.x * (256 / NCH) + slot; v < total; v += 4 * stride) {
      float x[4][8];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (v + u * stride < total) load8<FMT>(X, pos(v + u * stride), chunk, x[u]);
        else {
#pragma unroll
          for (int k = 0; k < 8; ++k) x[u][k] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int k = 0; k < 8; ++k) { s[k] += x[u][k]; q[k] = fmaf(x[u][k], x[u][k], q[k]); }
    }
  }
  // lanes with the same chunk are NCH apart: fold them with shuffles, then one shared-memory atomic per warp and channel
#pragma unroll
  for (int k = 0; k < 8; ++k)
    for (int o = NCH; o < 32; o <<= 1) { s[k] += __shfl_xor_sync(0xffffffffu, s[k], o); q[k] += __shfl_xor_sync(0xffffffffu, q[k], o); }
  if ((threadIdx.x & 31) < NCH && chunk * 8 < C) {
#pragma unroll
    for (int k = 0; k < 8; ++k) { atomicAdd(&red[chunk * 8 + k][0], s[k]); atomicAdd(&red[chunk * 8 + k][1], q[k]); }
  }
  __syncthreads();
  if (threadIdx.x < C) {
    atomicAdd(&sums[threadIdx.x * 2], (double)red[threadIdx.x][0]);
    atomicAdd(&sums[threadIdx.x * 2 + 1], (double)red[threadIdx.x][1]);
  }
}

// sums[kCountSlot] carries the element count when the sums are all-reduced over the ranks (synchronised BatchNorm)
constexpr int kCountSlot = 192;
constexpr int kSumsStride = 256;          // doubles per reduction buffer (one per layer and direction: a single memset clears them all)
__global__ void tset_count_kernel(double* __restrict__ sums, double count) { sums[kCountSlot] = count; }

// all-reduce the local BatchNorm sums (+ count) over the ranks through the caller's hook; `cnt` then points at the global count
static int sync_sums(sc_ctx* ctx, double* sums, double count, const double** cnt, cudaStream_t s) {
  *cnt = nullptr;
  if (!ctx->ar_hook) return SC_OK;
  tset_count_kernel<<<1, 1, 0, s>>>(sums, count);
  ctx->launches++;
  SC_CHECK(ctx->ar_hook(ctx->ar_user, sums, kCountSlot + 1, s) == 0, SC_ERR_STATE, "the all-reduce hook of sc_set_allreduce_hook failed");
  *cnt = sums + kCountSlot;
  return SC_OK;
}

// batch mean / inverse standard deviation of channel c from the reduction buffer (biased variance, eps 1e-4: Lasagne's BatchNormLayer)
__device__ __forceinline__ void bn_moments(const double* __restrict__ sums, double count, int c, float& mean, float& istd) {
  const double m = sums[c * 2] / count;
  double var = sums[c * 2 + 1] / count - m * m;
  if (var < 0) var = 0;
  mean = (float)m;
  istd = (float)(1.0 / sqrt(var + (double)kBnEps));
}
// Head of the activation kernels: the moments of all channels -> shared memory (one double division / square root per channel
// and CTA, then a barrier); the first CTA also publishes them for the backward pass and, through the gradient buffer, for the optimiser
__device__ __forceinline__ void bn_moments_cta(const double* __restrict__ sums, double count, int C, float (&s_mu)[64], float (&s_is)[64],
                                               float* __restrict__ mean, float* __restrict__ istd, float* __restrict__ g_mean_slot,
                                               float* __restrict__ g_istd_slot) {
  if (threadIdx.x < 64) {
    float m = 0.f, is = 0.f;
    if (threadIdx.x < C) {
      bn_moments(sums, count, threadIdx.x, m, is);
      if (blockIdx.x == 0) { mean[threadIdx.x] = m; istd[threadIdx.x] = is; g_mean_slot[threadIdx.x] = m; g_istd_slot[threadIdx.x] = is; }
    }
    s_mu[threadIdx.x] = m; s_is[threadIdx.x] = is;
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------------
// y = (x - mean) * gamma * istd + beta; a = prelu(y); optional 2x2 / 2 max-pool with arg-max record.
// Writes the activation map (pixel-major split, the next conv's input) and its planar transposed copy
// AT[2 * CP][Npix] (rows 0..CP-1 hi, CP..2CP-1 lo: the wgrad operand), zeros outside the valid region.
// One CTA = 64 consecutive positions of the OUTPUT map x all channel chunks.
// ---------------------------------------------------------------------------------------------------------------
template <int FMT>
__global__ void __launch_bounds__(64 * (FMT / 8), FMT == 32 ? 5 : 2) tbn_act_kernel(const float* __restrict__ X, int n, int C, int inPw, int inPitch,
                                                                  const double* __restrict__ sums, double count, const double* __restrict__ cnt,
                                                                  float* __restrict__ mean, float* __restrict__ istd,
                                                                  float* __restrict__ g_mean_slot, float* __restrict__ g_istd_slot,
                                                                  const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                  const float* __restrict__ alpha, int pool,
                                                                  float* __restrict__ A, int oR, int oPitch, int oH,
                                                                  uint8_t* __restrict__ idx, uint16_t* __restrict__ AT, int CP) {
  constexpr int NCH = FMT / 8;
  __shared__ uint16_t tile[2][FMT][66];
  __shared__ float s_mu[64], s_is[64];
  if (cnt) count = *cnt;
  bn_moments_cta(sums, count, C, s_mu, s_is, mean, istd, g_mean_slot, g_istd_slot);
  const int chunk = threadIdx.x % NCH, px = threadIdx.x / NCH;
  const int64_t oPw = (int64_t)n * oPitch, npix = (int64_t)oR * oPw;
  const int64_t q = (int64_t)blockIdx.x * 64 + px;
  float a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = 0.f;
  if (q < npix) {
    const int c = (int)(q % oPitch);
    const int s = (int)((q / oPitch) % n);
    const int r = (int)(q / oPw);
    const bool valid = r < oH && c < oH && chunk * 8 < C;
    uint32_t best = 0;      // 2 bits per channel
    if (valid) {
      float sc_[8], sh[8], al[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int ch = chunk * 8 + k;
        const bool on = ch < C;
        const float g = on ? gamma[ch] * s_is[ch] : 0.f;
        sc_[k] = g; sh[k] = on ? beta[ch] - s_mu[ch] * g : 0.f; al[k] = on ? alpha[ch] : 0.f;
      }
      if (!pool) {
        float x[8];
        load8<FMT>(X, (int64_t)r * inPw + (int64_t)s * inPitch + c, chunk, x);
#pragma unroll
        for (int k = 0; k < 8; ++k) a[k] = prelu(fmaf(x[k], sc_[k], sh[k]), al[k]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float x[8];
          load8<FMT>(X, (int64_t)(2 * r + (j >> 1)) * inPw + (int64_t)s * inPitch + 2 * c + (j & 1), chunk, x);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float y = prelu(fmaf(x[k], sc_[k], sh[k]), al[k]);
            if (j == 0 || y > a[k]) { a[k] = y; best = (best & ~(3u << (2 * k))) | ((uint32_t)j << (2 * k)); }
          }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (chunk * 8 + k >= C) a[k] = 0.f;
        if (idx) reinterpret_cast<uint16_t*>(idx)[q * NCH + chunk] = (uint16_t)best;
      }
    }
    uint4 h, l;
    split8(a, h, l);
    store8<FMT>(A, q, chunk, h, l);
    if (AT) {
      const uint32_t hh[4] = {h.x, h.y, h.z, h.w}, ll[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        tile[0][chunk * 8 + 2 * k][px] = (uint16_t)(hh[k] & 0xffffu); tile[0][chunk * 8 + 2 * k + 1][px] = (uint16_t)(hh[k] >> 16);
        tile[1][chunk * 8 + 2 * k][px] = (uint16_t)(ll[k] & 0xffffu); tile[1][chunk * 8 + 2 * k + 1][px] = (uint16_t)(ll[k] >> 16);
      }
    }
  } else if (AT) {
#pragma unroll
    for (int k = 0; k < 8; ++k) { tile[0][chunk * 8 + k][px] = 0; tile[1][chunk * 8 + k][px] = 0; }
  }
  if (!AT) return;       // the MN-major wgrad reads the pixel-major map itself: no planar transposed copy
  __syncthreads();
  {
    // rows of 64 positions (128 B) per channel: one warp per row, lane = two positions
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int64_t q0 = (int64_t)blockIdx.x * 64;
    for (int row = warp; row < 2 * CP; row += nw) {
      const int half = row / CP, ch = row - half * CP;
      const int64_t qa = q0 + 2 * lane;
      if (qa < npix) {   // npix is even
        const uint32_t v = (uint32_t)tile[half][ch][2 * lane] | ((uint32_t)tile[half][ch][2 * lane + 1] << 16);
        *reinterpret_cast<uint32_t*>(AT + (int64_t)row * npix + qa) = v;
      }
    }
  }
}

// conv5 activation (valid 3x3 of the [7][n][8] F64CH map) -> F5 [n][540] in (c, h, w) order with the l1drop mask applied
__global__ void tact5_flatten_kernel(const float* __restrict__ X4, int n, const double* __restrict__ sums, double count, const double* __restrict__ cnt,
                                     float* __restrict__ mean, float* __restrict__ istd, float* __restrict__ g_mean_slot, float* __restrict__ g_istd_slot,
                                     const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ alpha,
                                     const uint8_t* __restrict__ mask /*+ b*540, row stride 2700*/, float* __restrict__ F5) {
  __shared__ float s_mu[64], s_is[64];
  if (cnt) count = *cnt;
  bn_moments_cta(sums, count, 60, s_mu, s_is, mean, istd, g_mean_slot, g_istd_slot);
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)n * 540) return;
  const int i = (int)(e / 540), k = (int)(e - (int64_t)i * 540);
  const int c = k / 9, r = k - c * 9, h = r / 3, w = r - h * 3;
  const __nv_bfloat16* px = reinterpret_cast<const __nv_bfloat16*>(reinterpret_cast<const char*>(X4) + ((int64_t)h * n * 8 + (int64_t)i * 8 + w) * 256);
  const float x = __bfloat162float(px[c]) + __bfloat162float(px[64 + c]);
  const float g = gamma[c] * s_is[c];
  const float y = prelu(fmaf(x, g, beta[c] - s_mu[c] * g), alpha[c]);
  F5[e] = mask[(int64_t)i * 2700 + k] ? 2.f * y : 0.f;
}

// ---------------------------------------------------------------------------------------------------------------
// conv block backward.  Incoming gradient dA of the block's output: a split map at the pooled resolution (pool = 1,
// routed through idx) or at full resolution, or for conv5 the gradient of the flattened features (plain [n][540]).
//   pass 1: s[c] = {sum dy, sum dy * xhat, sum da * y * [y <= 0]}  with y = xhat * gamma + beta, dy = da * (y > 0 ? 1 : alpha)
//   pass 2: dx = gamma * istd * (dy - s1/m - xhat * s2/m)
// ---------------------------------------------------------------------------------------------------------------
template <int FMT, int DFMT>
__device__ __forceinline__ void bwd_point(const float* X, const float* dA, const uint8_t* idx, const float* dF5, int dF5_ld, const uint8_t* mask,
                                          int n, int C, int Pw, int pitch, int pool, int dPw, int dPitch, int r, int s, int c, int chunk,
                                          float (&x)[8], float (&g)[8]) {
  load8<FMT>(X, (int64_t)r * Pw + (int64_t)s * pitch + c, chunk, x);
  if (dF5) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int ch = chunk * 8 + k;
      const int f = ch * 9 + r * 3 + c;
      g[k] = (ch < C && mask[(int64_t)s * 2700 + f]) ? 2.f * dF5[(int64_t)s * dF5_ld + f] : 0.f;
    }
  } else if (pool) {
    const int64_t pq = (int64_t)(r >> 1) * dPw + (int64_t)s * dPitch + (c >> 1);
    float d[8];
    load8<DFMT>(dA, pq, chunk, d);
    const uint32_t best = reinterpret_cast<const uint16_t*>(idx)[pq * (FMT / 8) + chunk];
    const uint32_t me = (uint32_t)((r & 1) * 2 + (c & 1));
#pragma unroll
    for (int k = 0; k < 8; ++k) g[k] = ((best >> (2 * k)) & 3u) == me ? d[k] : 0.f;
  } else {
    load8<DFMT>(dA, (int64_t)r * dPw + (int64_t)s * dPitch + c, chunk, g);
  }
}

template <int FMT, int DFMT>
__global__ void __launch_bounds__(256) tbn_bwd_reduce_kernel(const float* __restrict__ X, const float* __restrict__ dA, const uint8_t* __restrict__ idx,
                                                             const float* __restrict__ dF5, int dF5_ld, const uint8_t* __restrict__ mask,
                                                             int n, int C, int H, int Pw, int pitch, int pool, int dPw, int dPitch,
                                                             const float* __restrict__ mean, const float* __restrict__ istd,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             const float* __restrict__ alpha, double* __restrict__ sums /*[64][3]*/) {
  constexpr int NCH = FMT / 8;
  __shared__ float red[64][3];
  for (int i = threadIdx.x; i < 192; i += 256) (&red[0][0])[i] = 0.f;
  __syncthreads();
  const int chunk = threadIdx.x % NCH, slot = threadIdx.x / NCH;
  const int64_t total = (int64_t)H * n * H;
  float s1[8], s2[8], s3[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s1[k] = s2[k] = s3[k] = 0.f;
  if (chunk * 8 < C) {
    float mu[8], is[8], ga[8], be[8], al[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int ch = chunk * 8 + k;
      const bool on = ch < C;
      mu[k] = on ? mean[ch] : 0.f; is[k] = on ? istd[ch] : 0.f; ga[k] = on ? gamma[ch] : 0.f; be[k] = on ? beta[ch] : 0.f; al[k] = on ? alpha[ch] : 0.f;
    }
for (int64_t v = (int64_t)blockIdx.x * (256 / NCH) + slot; v < total; v += (int64_t)gridDim.x * (256 / NCH)) {
      const int c = (int)(v % H);
      const int s = (int)((v / H) % n);
      const int r = (int)(v / ((int64_t)H * n));
      float x[8], g[8];
      bwd_point<FMT, DFMT>(X, dA, idx, dF5, dF5_ld, mask, n, C, Pw, pitch, pool, dPw, dPitch, r, s, c, chunk, x, g);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float xh = (x[k] - mu[k]) * is[k];
        const float yv = fmaf(xh, ga[k], be[k]);
        const float dy = yv > 0.f ? g[k] : al[k] * g[k];
        s1[k] += dy; s2[k] = fmaf(dy, xh, s2[k]);
        if (yv <= 0.f) s3[k] = fmaf(g[k], yv, s3[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k)
    for (int o = NCH; o < 32; o <<= 1) {
      s1[k] += __shfl_xor_sync(0xffffffffu, s1[k], o); s2[k] += __shfl_xor_sync(0xffffffffu, s2[k], o); s3[k] += __shfl_xor_sync(0xffffffffu, s3[k], o);
    }
  if ((threadIdx.x & 31) < NCH && chunk * 8 < C) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      atomicAdd(&red[chunk * 8 + k][0], s1[k]); atomicAdd(&red[chunk * 8 + k][1], s2[k]); atomicAdd(&red[chunk * 8 + k][2], s3[k]);
    }
  }
  __syncthreads();
  if (threadIdx.x < C) {
    atomicAdd(&sums[threadIdx.x * 3], (double)red[threadIdx.x][0]);
    atomicAdd(&sums[threadIdx.x * 3 + 1], (double)red[threadIdx.x][1]);
    atomicAdd(&sums[threadIdx.x * 3 + 2], (double)red[threadIdx.x][2]);
  }
}
// The beta / gamma / slope gradients are the three per-channel sums of pass 1 -- the LOCAL sums: the gradient all-reduce adds the
// ranks.  Without a synchronised-BatchNorm hook the first CTA of the pass-2 kernel writes them (gbeta != nullptr); with a hook the
// sums are all-reduced in place before pass 2, so this one-CTA kernel copies them out first.
__device__ __forceinline__ void bn_publish_grads(const double* __restrict__ sums, int C, float* __restrict__ gbeta, float* __restrict__ ggamma,
                                                 float* __restrict__ galpha) {
  if (gbeta && blockIdx.x == 0 && threadIdx.x < C) {
    const int c = threadIdx.x;
    gbeta[c] = (float)sums[c * 3]; ggamma[c] = (float)sums[c * 3 + 1]; galpha[c] = (float)sums[c * 3 + 2];
  }
}
__global__ void tbn_bwd_params_kernel(const double* __restrict__ sums, int C, float* __restrict__ gbeta, float* __restrict__ ggamma,
                                      float* __restrict__ galpha) {
  bn_publish_grads(sums, C, gbeta, ggamma, galpha);
}

// pass 2 over ALL positions of the conv-output map (64 consecutive positions per CTA):
//   frame   (l >= 1): dx as a split map of the same geometry, zeros outside the valid region = the dgrad sweep's input
//                     (the sweep reads it with a window offset of (-2, -2): full correlation, zero fill by the TMA unit)
//   DT      (l >= 1): three planar transposed copies [3][2 * CP][Npix], copy k shifted right by k positions
//                     (DT_k[p] = dx[p - k]), zeros outside the valid region = the wgrad operand of filter column k
//   planar  (l == 0): fp32 [n][C][H][ld] for the CUDA-core conv1 wgrad
template <int FMT, int DFMT>
__global__ void __launch_bounds__(64 * (FMT / 8), FMT == 32 ? 6 : 3) tbn_bwd_dx_kernel(const float* __restrict__ X, const float* __restrict__ dA, const uint8_t* __restrict__ idx,
                                                                     const float* __restrict__ dF5, int dF5_ld, const uint8_t* __restrict__ mask,
                                                                     int n, int C, int H, int R, int Pw, int pitch, int pool, int dPw, int dPitch,
                                                                     const float* __restrict__ mean, const float* __restrict__ istd,
                                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                     const float* __restrict__ alpha, const double* __restrict__ sums, double count,
                                                                     const double* __restrict__ cnt,
                                                                     float* __restrict__ gbeta, float* __restrict__ ggamma, float* __restrict__ galpha,
                                                                     float* __restrict__ frame, uint16_t* __restrict__ DT, int CP,
                                                                     float* __restrict__ planar, int pld) {
  constexpr int NCH = FMT / 8;
  if (cnt) count = *cnt;
  bn_publish_grads(sums, C, gbeta, ggamma, galpha);
  __shared__ uint16_t tile[2][FMT][68];     // columns 0..63: this CTA's positions; 64, 65: the two positions to their left
  // per-channel constants once per CTA: the two double divisions per channel cost more than the rest of a thread's work (issuing the
  // map loads before this barrier was tried: the longer live ranges cost more occupancy than the overlap gains)
  __shared__ float s_k[64][5];              // mean, istd, gamma, beta, alpha
  __shared__ float s_m[64][2];              // sum(dy) / m, sum(dy xhat) / m
  if (threadIdx.x < 64) {
    const int ch = threadIdx.x;
    const bool on = ch < C;
    s_k[ch][0] = on ? mean[ch] : 0.f; s_k[ch][1] = on ? istd[ch] : 0.f; s_k[ch][2] = on ? gamma[ch] : 0.f;
    s_k[ch][3] = on ? beta[ch] : 0.f; s_k[ch][4] = on ? alpha[ch] : 0.f;
    s_m[ch][0] = on ? (float)(sums[ch * 3] / count) : 0.f;
    s_m[ch][1] = on ? (float)(sums[ch * 3 + 1] / count) : 0.f;
  }
  __syncthreads();
  const int chunk = threadIdx.x % NCH, px = threadIdx.x / NCH;
  const int64_t npix = (int64_t)R * Pw;
  const int64_t q0 = (int64_t)blockIdx.x * 64;
  // dx of position q (zeros outside the valid region / the map) -> returns whether q is a valid position of this chunk
  auto point = [&](int64_t q, float (&dx)[8], int& r, int& s, int& c) {
#pragma unroll
    for (int k = 0; k < 8; ++k) dx[k] = 0.f;
    if (q < 0 || q >= npix) return false;
    c = (int)(q % pitch);
    s = (int)((q / pitch) % n);
    r = (int)(q / Pw);
    if (!(r < H && c < H && chunk * 8 < C)) return false;
    float x[8], g[8];
    bwd_point<FMT, DFMT>(X, dA, idx, dF5, dF5_ld, mask, n, C, Pw, pitch, pool, dPw, dPitch, r, s, c, chunk, x, g);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int ch = chunk * 8 + k;
      if (ch < C) {
        const float is = s_k[ch][1], ga = s_k[ch][2];
        const float xh = (x[k] - s_k[ch][0]) * is;
        const float yv = fmaf(xh, ga, s_k[ch][3]);
        const float dy = yv > 0.f ? g[k] : s_k[ch][4] * g[k];
        dx[k] = ga * is * (dy - s_m[ch][0] - xh * s_m[ch][1]);
      }
    }
    return true;
  };
  auto to_tile = [&](const uint4& h, const uint4& l, int col) {
    const uint32_t hh[4] = {h.x, h.y, h.z, h.w}, ll[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      tile[0][chunk * 8 + 2 * k][col] = (uint16_t)(hh[k] & 0xffffu); tile[0][chunk * 8 + 2 * k + 1][col] = (uint16_t)(hh[k] >> 16);
      tile[1][chunk * 8 + 2 * k][col] = (uint16_t)(ll[k] & 0xffffu); tile[1][chunk * 8 + 2 * k + 1][col] = (uint16_t)(ll[k] >> 16);
    }
  };
  const int64_t q = q0 + px;
  float dx[8];
  int r = 0, s = 0, c = 0;
  const bool valid = point(q, dx, r, s, c);
  if (planar) {
    if (valid) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int ch = chunk * 8 + k;
        if (ch < C) planar[(((int64_t)s * C + ch) * H + r) * pld + c] = dx[k];
      }
    }
    return;
  }
  uint4 h, l;
  split8(dx, h, l);
  if (q < npix) store8<FMT>(frame, q, chunk, h, l);
  if (!DT) return;       // wgrad reads the pixel-major frame itself (wgrad_mn_kernel): no planar copies
  to_tile(h, l, px);
  if (px < 2) {          // the shifted copies of this CTA's 64 positions start one / two positions to the left: recompute those two
    float dh[8];
    int r2, s2, c2;
    point(q0 - 2 + px, dh, r2, s2, c2);
    uint4 h2, l2;
    split8(dh, h2, l2);
    to_tile(h2, l2, 64 + px);
  }
  __syncthreads();
  // DT_k[p] = dx[p - k]: every copy is written as whole aligned 128 B rows (two positions per lane)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int64_t qa = q0 + 2 * lane;
  if (qa < npix) {     // npix is even
    for (int row = warp; row < 2 * CP; row += nw) {
      const int half = row / CP, ch = row - half * CP;
      const uint16_t* t = tile[half][ch];
      const uint32_t m2 = lane ? t[2 * lane - 2] : t[64], m1 = lane ? t[2 * lane - 1] : t[65], v0 = t[2 * lane], v1 = t[2 * lane + 1];
      *reinterpret_cast<uint32_t*>(DT + (int64_t)row * npix + qa) = v0 | (v1 << 16);
      *reinterpret_cast<uint32_t*>(DT + ((int64_t)2 * CP + row) * npix + qa) = m1 | (v0 << 16);
      *reinterpret_cast<uint32_t*>(DT + ((int64_t)4 * CP + row) * npix + qa) = m2 | (m1 << 16);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// conv1 backward in one pass: dx of the BatchNorm / PReLU block and, fused, the conv1 weight gradient (1 -> 20 channels,
// K = 9: CUDA cores).  gW[co][8 - t] += sum over pixels dx[co] * patch[r + ky][c + kx]; 72 accumulators per thread (8 channels
// x 9 taps), folded with shuffles and shared-memory atomics.  conv1 has no dgrad, so dx is never written.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 2) tbn_bwd_conv1_kernel(const float* __restrict__ X, const float* __restrict__ dA, const float* __restrict__ patches,
                                                            int n, const float* __restrict__ mean, const float* __restrict__ istd,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            const float* __restrict__ alpha, const double* __restrict__ sums, double count,
                                                            const double* __restrict__ cnt, float* __restrict__ gbeta, float* __restrict__ ggamma,
                                                            float* __restrict__ galpha, float* __restrict__ gW) {
  constexpr int C = 20, H = 30;
  if (cnt) count = *cnt;
  bn_publish_grads(sums, C, gbeta, ggamma, galpha);
  __shared__ float red[24][9];
  for (int i = threadIdx.x; i < 24 * 9; i += 256) (&red[0][0])[i] = 0.f;
  __syncthreads();
  const int chunk = threadIdx.x & 3, slot = threadIdx.x >> 2;
  const int Pw = n * 32;
  float acc[8][9];
#pragma unroll
  for (int k = 0; k < 8; ++k)
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[k][t] = 0.f;
  // per-channel constants in shared memory (7 x 8 registers less per thread: two CTAs fit an SM instead of one)
  __shared__ float s_c[24][8];              // mean, istd, gamma, beta, alpha, sum(dy) / m, sum(dy xhat) / m, gamma * istd
  if (threadIdx.x < 24) {
    const int ch = threadIdx.x;
    const bool on = ch < C;
    s_c[ch][0] = on ? mean[ch] : 0.f; s_c[ch][1] = on ? istd[ch] : 0.f; s_c[ch][2] = on ? gamma[ch] : 0.f;
    s_c[ch][3] = on ? beta[ch] : 0.f; s_c[ch][4] = on ? alpha[ch] : 0.f;
    s_c[ch][5] = on ? (float)(sums[ch * 3] / count) : 0.f; s_c[ch][6] = on ? (float)(sums[ch * 3 + 1] / count) : 0.f;
    s_c[ch][7] = on ? gamma[ch] * istd[ch] : 0.f;
  }
  __syncthreads();
  if (chunk < 3) {
    const int64_t total = (int64_t)H * n * H;
    for (int64_t v = (int64_t)blockIdx.x * 64 + slot; v < total; v += (int64_t)gridDim.x * 64) {
      const int c = (int)(v % H);
      const int s = (int)((v / H) % n);
      const int r = (int)(v / ((int64_t)H * n));
      const int64_t p = (int64_t)r * Pw + (int64_t)s * 32 + c;
      float x[8], g[8];
      load8<32>(X, p, chunk, x);
      load8<32>(dA, p, chunk, g);
      const float* src = patches + (int64_t)s * 1024 + r * 32 + c;
      float w[9];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) w[ky * 3 + kx] = __ldg(src + ky * 32 + kx);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float4 c0 = *reinterpret_cast<const float4*>(&s_c[chunk * 8 + k][0]);     // mean, istd, gamma, beta
        const float4 c1 = *reinterpret_cast<const float4*>(&s_c[chunk * 8 + k][4]);     // alpha, m1, m2, gamma * istd
        const float xh = (x[k] - c0.x) * c0.y;
        const float yv = fmaf(xh, c0.z, c0.w);
        const float dy = yv > 0.f ? g[k] : c1.x * g[k];
        const float dx = c0.z * c0.y * (dy - c1.y - xh * c1.z);
#pragma unroll
        for (int t = 0; t < 9; ++t) acc[k][t] = fmaf(dx, w[t], acc[k][t]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k)
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      float v = acc[k][t];
      v += __shfl_xor_sync(0xffffffffu, v, 4); v += __shfl_xor_sync(0xffffffffu, v, 8); v += __shfl_xor_sync(0xffffffffu, v, 16);
      if ((threadIdx.x & 31) < 3) atomicAdd(&red[chunk * 8 + k][t], v);
    }
  __syncthreads();
  for (int i = threadIdx.x; i < C * 9; i += 256) {
    const int co = i / 9, t = i - co * 9;
    atomicAdd(&gW[co * 9 + (8 - t)], red[co][t]);     // correlation tap t = element 8 - t of the (true-convolution) filter
  }
}

// ---------------------------------------------------------------------------------------------------------------
// wgrad on the tensor cores.  With p' = p + tx:
//   gW[ty][tx][ci][co] = sum_p A[ci][p + ty*Pw + tx] * dX[co][p] = sum_p' A[ci][p' + ty*Pw] * DT_tx[co][p']
//   A operand (M): the three row-shifted windows of the planar input map, stacked: 3 x CIN8 <= 120 rows of one M = 128 tile
//   B operand (N): the three column-shifted copies DT_tx of the planar output gradient stacked, 3 x NCO rows: ONE MMA per
//                   k-step and split term produces all three filter columns (the A tile is fetched once instead of thrice)
//   K: 64 pixels per stage; the CTAs split the pixel range (split-K) and add their partial sums atomically
// warp 0: TMA producer (12 boxes per stage), warp 1: MMA issue (3 accumulators x 4 k-steps x 3 split products), warps 2-5: epilogue
// ---------------------------------------------------------------------------------------------------------------
static inline int pad8(int c) { return (c + 7) & ~7; }
static inline int pad16(int c) { return (c + 15) & ~15; }

struct WgradArgs {
  int cin, cout, cin8, nco;      // real channels, input rows per window (multiple of 8), gradient rows per copy in shared memory (multiple of 16)
  int co8;                       // gradient rows per copy as stored / loaded (multiple of 8): the rows [co8, nco) of a slot are never
                                 // written and only feed accumulator columns nobody reads
  int Pw;                        // wide-row pitch in pixels: filter row = shift by Pw
  int nkb;                       // 64-pixel blocks to reduce over
  int stages;
  float* gW;                     // [cout][cin][3][3] master-layout gradient (accumulated atomically)
};

__global__ void __launch_bounds__(192, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapD, const WgradArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int a_half = 3 * a.cin8 * 128;                    // bytes of the stacked hi (or lo) windows
  const int d_one = a.nco * 128, d_half = 3 * d_one;      // one shifted copy; the three hi (or lo) copies
  const int stage_bytes = 2 * a_half + 2 * d_half;        // (the M = 128 tile of the lo windows reads on into the gradient boxes)
  const int tx_bytes = 2 * a_half + 2 * 3 * a.co8 * 128;  // bytes the TMA unit actually delivers per stage
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + a.stages * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + a.stages;
  uint64_t* done = bars + 2 * a.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // this CTA's share of the pixel blocks
  const int per = (a.nkb + gridDim.x - 1) / gridDim.x;
  const int kb0 = blockIdx.x * per, kb1 = min(a.nkb, kb0 + per);
  const int nk = kb1 - kb0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (nk > 0) {
    if (warp == 0) {
      if (lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapD)) : "memory");
        for (int i = 0; i < nk; ++i) {
          const int s = i % a.stages, use = i / a.stages;
          if (use > 0) mbar_wait(&empty[s], (use - 1) & 1);
          mbar_expect_tx(&full[s], (uint32_t)tx_bytes);
          uint8_t* sp = smem + s * stage_bytes;
          const int p0 = (kb0 + i) * 64;
#pragma unroll 1
          for (int t = 0; t < 3; ++t) {
            tma_load_2d(&mapA, &full[s], sp + t * a.cin8 * 128, p0 + t * a.Pw, 0);                 // window of filter row t, hi rows
            tma_load_2d(&mapA, &full[s], sp + a_half + t * a.cin8 * 128, p0 + t * a.Pw, a.cin8);   // lo rows
            tma_load_2d(&mapD, &full[s], sp + 2 * a_half + t * d_one, p0, t * 2 * a.co8);          // copy shifted by t, hi rows
            tma_load_2d(&mapD, &full[s], sp + 2 * a_half + d_half + t * d_one, p0, t * 2 * a.co8 + a.co8);
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      const uint32_t leader = elect_one();
      // D = F32, A = B = BF16, both K-major, N = 3 * nco (the three shifted copies are adjacent row blocks), M = 128
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((3 * a.nco) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      for (int i = 0; i < nk; ++i) {
        const int s = i % a.stages;
        mbar_wait(&full[s], (i / a.stages) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sp = smem_u32(smem + s * stage_bytes);
        const uint64_t ah = umma_desc(sp), al = umma_desc(sp + a_half);
        const uint64_t dh = umma_desc(sp + 2 * a_half), dl = umma_desc(sp + 2 * a_half + d_half);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint64_t o = (uint64_t)(j * 2);
          umma_bf16_elect(tmem_base, al + o, dh + o, idesc, (i | j) != 0, leader);
          umma_bf16_elect(tmem_base, ah + o, dl + o, idesc, 1, leader);
          umma_bf16_elect(tmem_base, ah + o, dh + o, idesc, 1, leader);
        }
        if (leader) umma_commit(&empty[s]);
        __syncwarp();
      }
      if (leader) umma_commit(done);
      __syncwarp();
    } else {
      const int q = warp & 3;      // TMEM lane quarter this warp may read
      mbar_wait(done, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int row = q * 32 + lane;
      const int ty = row / a.cin8, ci = row - ty * a.cin8;
      const bool on = ty < 3 && ci < a.cin;
      for (int tx = 0; tx < 3; ++tx) {
        for (int c0 = 0; c0 < a.nco; c0 += 16) {
          uint32_t rr[16];
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(tx * a.nco + c0);
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
              : "=r"(rr[0]), "=r"(rr[1]), "=r"(rr[2]), "=r"(rr[3]), "=r"(rr[4]), "=r"(rr[5]), "=r"(rr[6]), "=r"(rr[7]), "=r"(rr[8]),
                "=r"(rr[9]), "=r"(rr[10]), "=r"(rr[11]), "=r"(rr[12]), "=r"(rr[13]), "=r"(rr[14]), "=r"(rr[15])
              : "r"(taddr));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (on) {
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const int co = c0 + k;
              // tap t of the correlation = element 8 - t of the (true-convolution) filter
              if (co < a.cout) atomicAdd(a.gW + ((int64_t)co * a.cin + ci) * 9 + (8 - (ty * 3 + tx)), __uint_as_float(rr[k]));
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256) : "memory");
  }
}

static int launch_wgrad_tc(sc_ctx* ctx, const uint16_t* AT, const uint16_t* DT, int cin, int cout, int cin8, int nco, int Pw, int64_t npix,
                           int rows_valid, float* gW, cudaStream_t st) {
  TcState* s = reinterpret_cast<TcState*>(ctx->tc_state);
  SC_CHECK(s != nullptr, SC_ERR_UNSUPPORTED, "tcgen05 back-end not initialised");
  SC_CHECK(npix % 8 == 0 && Pw % 8 == 0 && npix < (1ll << 31), SC_ERR_ARG, "wgrad_tc: bad map size");
  SC_CHECK(3 * cin8 <= 128 && nco <= 64 && nco % 16 == 0 && cin8 % 8 == 0, SC_ERR_ARG, "wgrad_tc: bad channel geometry");
  WgradArgs a;
  a.cin = cin; a.cout = cout; a.cin8 = cin8; a.nco = nco; a.Pw = Pw; a.gW = gW;
  a.co8 = pad8(cout);
  a.nkb = (int)(((int64_t)rows_valid * Pw + 2 + 63) / 64);  // the (shifted) gradient is zero beyond its valid rows
  const int stage_bytes = 2 * 3 * cin8 * 128 + 2 * 3 * nco * 128;
  a.stages = (227 * 1024 - 2048) / stage_bytes;
  if (a.stages > 6) a.stages = 6;
  SC_CHECK(a.stages >= 2, SC_ERR_ARG, "wgrad_tc: stage does not fit (%d bytes)", stage_bytes);
  const size_t smem = 1024 + (size_t)a.stages * stage_bytes + (2 * a.stages + 1) * 8 + 16;
  CUtensorMap mapA, mapD;
  {
    cuuint64_t dims[2] = {(cuuint64_t)npix, (cuuint64_t)(2 * cin8)};
    cuuint64_t strides[1] = {(cuuint64_t)npix * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)cin8};
    cuuint32_t es[2] = {1, 1};
    CUresult r = s->encode(&mapA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(AT), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "wgrad_tc: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)npix, (cuuint64_t)(3 * 2 * a.co8)};
    cuuint64_t strides[1] = {(cuuint64_t)npix * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)a.co8};
    cuuint32_t es[2] = {1, 1};
    CUresult r = s->encode(&mapD, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(DT), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "wgrad_tc: cuTensorMapEncodeTiled(D) failed with %d", (int)r);
  }
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(wgrad_tc_kernel), 227 * 1024));
  // at least ~6 pixel blocks per CTA: the epilogue (up to 120 x 3 x 60 atomics per CTA) must not dominate
  int grid = (a.nkb + 5) / 6;
  if (grid > ctx->sm_count) grid = ctx->sm_count;
  if (grid < 1) grid = 1;
  ProfScope prof(ctx, PC_TRAIN_BWD, st);
  wgrad_tc_kernel<<<grid, 192, smem, st>>>(mapA, mapD, a);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// wgrad straight from the PIXEL-major split maps (no planar copies): both operands MN-major.
//   gW[ty][tx][ci][co] = sum_p A[p + ty*Pw + tx][ci] * dX[p][co]
// A TMA box of 64 bf16 x 64 pixels of a split map is, in shared memory, 64 K-rows (pixels) of 128 B holding 64 "MN" elements:
// exactly the canonical MN-major SWIZZLE_128B operand (8-row groups 1024 B apart = SBO; further 64-element MN chunks LBO apart).
// The 64 MN elements of a 128 B pixel (20-channel maps) are [32 hi | 32 lo]; a 256 B pixel gives a hi box and a lo box = M (or N) 128.
// ONE MMA per k-step then produces all four hi/lo blocks of the product; the epilogue adds hi*hi + hi*lo + lo*hi and drops lo*lo.
// A tap is a shift of the OUTER (pixel) TMA coordinate by ty*Pw + tx: any integer, so the three column taps need no shifted copies.
//   blockIdx.y = filter row ty; the CTAs of a row split the pixel range (split-K) and add their partial sums atomically
//   128 B input pixels: M = 128 stacks two column taps (tx, tx + 1); 256 B input pixels: M = 128 = hi | lo of one column tap
// warp 0: TMA producer, warp 1: MMA issue, warps 2-5: epilogue
// ---------------------------------------------------------------------------------------------------------------
struct WgradMnArgs {
  int cin, cout;
  int nbA, nbD;                  // boxes per pixel of the input map / the gradient map (1: 128 B pixels, 2: 256 B pixels = hi box + lo box)
  int Pw;                        // wide-row pitch in pixels
  int kp;                        // pixels per pipeline stage (multiple of 16, <= 192): one TMA box of kp (+ 2) pixel rows per hi / lo half
  int win_bytes, box_bytes;      // shared-memory bytes reserved per input window ((kp + 2) x 128 B, 1024-aligned) / per gradient box (kp x 128 B)
  int nkb;                       // kp-pixel blocks to reduce over
  int stages;
  float* gW;                     // [cout][cin][3][3] master-layout gradient (accumulated atomically)
};

// MN-major, SWIZZLE_128B: SBO = 8 pixel rows (1024 B); LBO = distance of the second 64-element MN chunk
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

__global__ void __launch_bounds__(192, 1)
wgrad_mn_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapD, const WgradMnArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // per stage: the input window of kp + 2 pixels (one box per hi / lo half) serves the three column taps -- a tap is a start address
  // shifted by whole 128 B pixel rows (the swizzle follows the absolute address bits) -- then the gradient boxes
  const int WG_WIN = a.win_bytes, WG_BOX = a.box_bytes;
  const int a_bytes = a.nbA * WG_WIN, d_bytes = a.nbD * WG_BOX;
  const int stage_bytes = a_bytes + d_bytes;
  const int ngroups = a.nbA == 1 ? 2 : 3;                                 // MMAs per k-step (accumulators)
  const int N = 64 * a.nbD;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + a.stages * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + a.stages;
  uint64_t* done = bars + 2 * a.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ty = blockIdx.y;
  const int per = (a.nkb + gridDim.x - 1) / gridDim.x;
  const int kb0 = blockIdx.x * per, kb1 = min(a.nkb, kb0 + per);
  const int nk = kb1 - kb0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (nk > 0) {
    if (warp == 0) {
      if (lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapD)) : "memory");
        for (int i = 0; i < nk; ++i) {
          const int s = i % a.stages, use = i / a.stages;
          if (use > 0) mbar_wait(&empty[s], (use - 1) & 1);
          mbar_expect_tx(&full[s], (uint32_t)(a.nbA * (a.kp + 2) * 128 + d_bytes));
          uint8_t* sp = smem + s * stage_bytes;
          const int p0 = (kb0 + i) * a.kp;
          for (int h = 0; h < a.nbA; ++h)        // pixels p0 + ty * Pw ... + kp + 1 (zero fill beyond the map)
            tma_load_2d(&mapA, &full[s], sp + h * WG_WIN, h * 64, p0 + ty * a.Pw);
          for (int h = 0; h < a.nbD; ++h) tma_load_2d(&mapD, &full[s], sp + a_bytes + h * WG_BOX, h * 64, p0);
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      const uint32_t leader = elect_one();
      // D = F32, A = B = BF16, both MN-major (bits 15, 16), N = 64 * nbD, M = 128
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      for (int i = 0; i < nk; ++i) {
        const int s = i % a.stages;
        mbar_wait(&full[s], (i / a.stages) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sp = smem_u32(smem + s * stage_bytes);
        const uint64_t dd = umma_desc_mn(sp + a_bytes, WG_BOX);
        // 256 B pixels: M = hi box | lo box of column tap g (start shifted by g rows)
        // 128 B pixels: M = column taps (2g, 2g + 1): the second chunk is the same window one pixel row further
        // (descriptors once per stage: the issue loop itself is two or three MMAs and one 64-bit add per k-step)
        const uint64_t ad0 = a.nbA == 2 ? umma_desc_mn(sp, WG_WIN) : umma_desc_mn(sp, 128);
        const uint64_t ad1 = a.nbA == 2 ? umma_desc_mn(sp + 128, WG_WIN) : umma_desc_mn(sp + 256, 128);
        const uint64_t ad2 = umma_desc_mn(sp + 256, WG_WIN);
        const uint32_t third = (leader && ngroups == 3) ? 1u : 0u;
        const int nks = a.kp >> 4;
        uint64_t o = 0;
#pragma unroll 4
        for (int j = 0; j < nks; ++j, o += (uint64_t)(2048 >> 4)) {      // 16 pixels = two 8-row groups = 2048 B per k-step
          const uint32_t acc = (i | j) != 0;
          umma_bf16_elect(tmem_base, ad0 + o, dd + o, idesc, acc, leader);
          umma_bf16_elect(tmem_base + (uint32_t)N, ad1 + o, dd + o, idesc, acc, leader);
          umma_bf16_elect(tmem_base + (uint32_t)(2 * N), ad2 + o, dd + o, idesc, acc, third);
        }
        if (leader) umma_commit(&empty[s]);
        __syncwarp();
      }
      if (leader) umma_commit(done);
      __syncwarp();
    } else {
      const int q = warp & 3;      // TMEM lane quarter this warp may read
      mbar_wait(done, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int row = q * 32 + lane;
      const int halfN = N >> 1;    // columns [0, halfN): hi parts of the gradient channels, [halfN, N): lo parts
      for (int g = 0; g < ngroups; ++g) {
        // accumulator row -> (column tap, input channel, hi / lo)
        int tx, ci; bool lo_row;
        if (a.nbA == 1) { tx = 2 * g + (row >> 6); const int r = row & 63; lo_row = r >= 32; ci = r & 31; }
        else { tx = g; lo_row = row >= 64; ci = row & 63; }
        const bool on = tx < 3 && ci < a.cin;
        for (int c0 = 0; c0 < halfN; c0 += 16) {
          uint32_t rh[16], rl[16];
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * N + c0);
          tmem_ld16_raw(taddr, rh);
          tmem_ld16_raw(taddr + (uint32_t)halfN, rl);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (on) {
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const int co = c0 + k;
              // hi row: hi*hi + hi*lo; lo row: lo*hi only.  tap t of the correlation = element 8 - t of the (true-convolution) filter
              const float v = lo_row ? __uint_as_float(rh[k]) : __uint_as_float(rh[k]) + __uint_as_float(rl[k]);
              if (co < a.cout) atomicAdd(a.gW + ((int64_t)co * a.cin + ci) * 9 + (8 - (ty * 3 + tx)), v);
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// A: the input activation map of the layer (fmtA = 32 / 64 channel slots per pixel), D: the zero-framed output gradient (fmtD)
static int launch_wgrad_mn(sc_ctx* ctx, const float* A, int fmtA, const float* D, int fmtD, int cin, int cout, int Pw, int64_t npix, int rows_valid,
                           float* gW, cudaStream_t st) {
  TcState* s = reinterpret_cast<TcState*>(ctx->tc_state);
  SC_CHECK(s != nullptr, SC_ERR_UNSUPPORTED, "tcgen05 back-end not initialised");
  SC_CHECK(npix < (1ll << 31) && cin <= fmtA && cout <= fmtD, SC_ERR_ARG, "wgrad_mn: bad geometry");
  WgradMnArgs a;
  a.cin = cin; a.cout = cout; a.nbA = fmtA == 32 ? 1 : 2; a.nbD = fmtD == 32 ? 1 : 2; a.Pw = Pw; a.gW = gW;
  // pixels per stage: long enough to amortise the per-stage hand-offs, short enough for >= 3 stages
  a.kp = (a.nbA == 1 && a.nbD == 1) ? 192 : 128;
  a.win_bytes = ((a.kp + 2) * 128 + 1023) & ~1023;
  a.box_bytes = a.kp * 128;
  a.nkb = (int)(((int64_t)rows_valid * Pw + a.kp - 1) / a.kp);      // the gradient is zero beyond its valid rows
  const int stage_bytes = a.nbA * a.win_bytes + a.nbD * a.box_bytes;
  a.stages = (227 * 1024 - 2048) / stage_bytes;
  if (a.stages > 6) a.stages = 6;
  SC_CHECK(a.stages >= 2, SC_ERR_ARG, "wgrad_mn: stage does not fit (%d bytes)", stage_bytes);
  const size_t smem = 1024 + (size_t)a.stages * stage_bytes + (2 * a.stages + 1) * 8 + 16;
  CUtensorMap mapA, mapD;
  auto encode = [&](CUtensorMap* m, const float* base, int fmt, int box_px) {
    cuuint64_t dims[2] = {(cuuint64_t)(2 * fmt), (cuuint64_t)npix};          // bf16 elements per pixel (hi | lo), pixels
    cuuint64_t strides[1] = {(cuuint64_t)fmt * 4};
    cuuint32_t box[2] = {64, (cuuint32_t)box_px};
    cuuint32_t es[2] = {1, 1};
    return s->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  };
  CUresult r = encode(&mapA, A, fmtA, a.kp + 2);        // kp pixels + the two further ones the column taps 1, 2 reach
  SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "wgrad_mn: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
  r = encode(&mapD, D, fmtD, a.kp);
  SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "wgrad_mn: cuTensorMapEncodeTiled(D) failed with %d", (int)r);
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(wgrad_mn_kernel), 227 * 1024));
  // split-K: three filter rows x gx CTAs, at least ~3 stages of pixels per CTA (the epilogue's atomics must not dominate)
  int gx = (a.nkb + 2) / 3;
  if (gx > ctx->sm_count / 3) gx = ctx->sm_count / 3;
  if (gx < 1) gx = 1;
  ProfScope prof(ctx, PC_TRAIN_BWD, st);
  wgrad_mn_kernel<<<dim3(gx, 3), 192, smem, st>>>(mapA, mapD, a);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// the convolutional part of the step for one branch
// ---------------------------------------------------------------------------------------------------------------
struct TLayer { int cin, cout, R, pitch, fmt, H, pool, oR, oPitch, oH; };
static const TLayer kTL[5] = {
    {1, 20, 30, 32, 32, 30, 0, 30, 32, 30},
    {20, 20, 30, 32, 32, 28, 1, 15, 16, 14},
    {20, 40, 15, 16, 64, 12, 0, 15, 16, 12},
    {40, 40, 15, 16, 64, 10, 1, 7, 8, 5},
    {40, 60, 7, 8, 64, 3, 0, 0, 0, 0},
};

size_t tc_branch_bytes(int n) {
  size_t b = 0;
  auto al = [](size_t v) { return (v + 1023) & ~(size_t)1023; };
  for (int l = 0; l < 5; ++l) {
    const TLayer& L = kTL[l];
    const size_t npx = (size_t)L.R * n * L.pitch;
    b += al(npx * L.fmt * 4);                                      // X_l
    if (l < 4) {
      const size_t opx = (size_t)L.oR * n * L.oPitch;
      b += al(opx * L.fmt * 4);                                    // A_l
      b += al(opx * 2 * pad8(L.cout) * 2);                         // A_l planar transposed (hi | lo)
      if (L.pool) b += al(opx * (L.fmt / 8) * 2);                  // arg-max record
    }
    b += 2 * 1024;                                                 // mean, istd
  }
  const size_t big32 = (size_t)30 * n * 32 * 128, big64 = (size_t)15 * n * 16 * 256;
  const size_t big = big32 > big64 ? big32 : big64;
  b += 2 * al(big);                                                // frame, dA
  b += al((size_t)30 * n * 32 * 3 * 2 * 32 * 2);                   // DT: three shifted copies (largest: conv2, 3 x 2 x 32 rows)
  b += al((size_t)n * 20 * 30 * 32 * 4);                           // planar fp32 dX of conv1
  b += al(10 * kSumsStride * 8) + 1024 * 4;                        // BatchNorm reduction buffers
  return b;
}

int tc_carve_branch(TcBranchBuf& T, char* base, int n) {
  size_t off = 0;
  auto take = [&](size_t bytes) { char* p = base + off; off += (bytes + 1023) & ~(size_t)1023; return p; };
  for (int l = 0; l < 5; ++l) {
    const TLayer& L = kTL[l];
    const size_t npx = (size_t)L.R * n * L.pitch;
    T.X[l] = reinterpret_cast<float*>(take(npx * L.fmt * 4));
    if (l < 4) {
      const size_t opx = (size_t)L.oR * n * L.oPitch;
      T.A[l] = reinterpret_cast<float*>(take(opx * L.fmt * 4));
      T.AT[l] = reinterpret_cast<uint16_t*>(take(opx * 2 * pad8(L.cout) * 2));
      T.idx[l] = L.pool ? reinterpret_cast<uint8_t*>(take(opx * (L.fmt / 8) * 2)) : nullptr;
    } else {
      T.A[l] = nullptr; T.AT[l] = nullptr; T.idx[l] = nullptr;
    }
    T.mean[l] = reinterpret_cast<float*>(take(256));
    T.istd[l] = reinterpret_cast<float*>(take(256));
  }
  const size_t big32 = (size_t)30 * n * 32 * 128, big64 = (size_t)15 * n * 16 * 256;
  const size_t big = big32 > big64 ? big32 : big64;
  T.frame = reinterpret_cast<float*>(take(big));
  T.dA = reinterpret_cast<float*>(take(big));
  T.DT = reinterpret_cast<uint16_t*>(take((size_t)30 * n * 32 * 3 * 2 * 32 * 2));
  T.dX0 = reinterpret_cast<float*>(take((size_t)n * 20 * 30 * 32 * 4));
  T.sums = reinterpret_cast<double*>(take(10 * kSumsStride * 8));   // per layer, forward (l) and backward (5 + l): [64][3] sums + the count slot
  return (int)0;
}

static unsigned cap_grid(sc_ctx* ctx, int64_t blocks, int per_sm) {
  const int64_t cap = (int64_t)ctx->sm_count * per_sm;
  return (unsigned)(blocks < 1 ? 1 : (blocks < cap ? blocks : cap));
}

// persistent buffers of the re-derived sweep panels: [branch][layer 1..4][fwd | dgrad] x (plain, pair)
static int ensure_train_panels(sc_ctx* ctx) {
  if (ctx->train_panels) return SC_OK;
  size_t total = 0;
  for (int l = 1; l < 5; ++l)
    for (int d = 0; d < 2; ++d) {
      const int kin = d ? kTL[l].cout : kTL[l].cin, nout = d ? kTL[l].cin : kTL[l].cout;
      const int ksteps = (kin + 15) / 16, bn = pad16(nout), npanels = (3 * ksteps + 3) / 4;
      total += 2 * (((size_t)npanels * 6 * bn * 64 * 2 + 1023) & ~(size_t)1023);
    }
  total *= 3;
  SC_CUDA(cudaMalloc(&ctx->train_panels, total));
  SC_CUDA(cudaMemset(ctx->train_panels, 0, total));        // the channel / k padding stays zero for good
  char* p = reinterpret_cast<char*>(ctx->train_panels);
  for (int b = 0; b < 3; ++b)
    for (int l = 1; l < 5; ++l)
      for (int d = 0; d < 2; ++d) {
        const int kin = d ? kTL[l].cout : kTL[l].cin, nout = d ? kTL[l].cin : kTL[l].cout;
        SweepW& S = ctx->train_sw[b][l][d];
        S.ksteps = (kin + 15) / 16; S.bn = pad16(nout); S.npanels = (3 * S.ksteps + 3) / 4;
        const size_t bytes = ((size_t)S.npanels * 6 * S.bn * 64 * 2 + 1023) & ~(size_t)1023;
        S.panels = reinterpret_cast<float*>(p); p += bytes;
        S.panels_pair = reinterpret_cast<float*>(p); p += bytes;
        S.scale = ctx->train_consts; S.shift = ctx->train_consts + kTrainZeros; S.alpha = ctx->train_consts;   // identity epilogue
      }
  return SC_OK;
}

int tc_train_prepare(sc_ctx* ctx) { return ensure_train_panels(ctx); }

int tc_branch_forward(sc_ctx* ctx, int b, const TcBranchBuf& T, const float* patches, const float* wf0, int n, const uint8_t* masks,
                      float* F5, cudaStream_t s) {
  SC_TRY(ensure_train_panels(ctx));
  const ParamOff& O = ctx->off;
  const BranchOff& Ob = O.br[b];
  float* P = ctx->params;
  float* G = ctx->grads;
  {
    PanelJobs jobs;
    int most = 0;
    for (int l = 1; l < 5; ++l)
      for (int d = 0; d < 2; ++d) {
        const SweepW& S = ctx->train_sw[b][l][d];
        jobs.j[(l - 1) * 2 + d] = {P + Ob.convW[l], kTL[l].cout, kTL[l].cin, d, S.ksteps, S.bn, reinterpret_cast<uint16_t*>(S.panels),
                                   reinterpret_cast<uint16_t*>(S.panels_pair)};
        const int ne = kTL[l].cout * kTL[l].cin * 9;
        most = ne > most ? ne : most;
      }
    derive_panels_kernel<<<dim3((most + 255) / 256, 8), 256, 0, s>>>(jobs);
    ctx->launches++;
  }
  SC_CUDA(cudaMemsetAsync(T.sums, 0, 10 * kSumsStride * sizeof(double), s));     // every BatchNorm reduction buffer of the step
  for (int l = 0; l < 5; ++l) {
    const TLayer& L = kTL[l];
    const int Pw = n * L.pitch;
    double* sums = T.sums + l * kSumsStride;
    const int64_t vpix = (int64_t)L.H * n * L.H;
    if (l == 0) {
      {
        ProfScope prof(ctx, PC_TRAIN_FWD, s);
        tconv1_kernel<<<cap_grid(ctx, ((int64_t)30 * n * 32 + 255) / 256, 8), 256, 0, s>>>(patches, n, wf0, T.X[0]);
      }
      tbn_stats_kernel<32><<<cap_grid(ctx, (vpix + 63) / 64 / 4 + 1, 2), 256, 0, s>>>(T.X[l], n, L.cout, L.H, Pw, L.pitch, sums);
      ctx->launches += 2;
    } else {
      // conv2..conv5: the sweep's epilogue accumulates the batch statistics of its raw output (no separate pass over the map)
      const TLayer& Li = kTL[l - 1];
      // With a synchronised-BatchNorm hook the statistics come from a separate pass over the STORED map instead (double sums of
      // identical values: N ranks then reproduce one rank up to the order of a handful of double additions).
      const SweepStats st = {sums, L.H, L.pitch};
      const bool fuse = ctx->train_fused_stats && !ctx->ar_hook;
      SC_TRY(launch_conv_sweep(ctx, ctx->train_sw[b][l][0], l, T.A[l - 1], Li.fmt == 32 ? 1 : 0, T.X[l], L.fmt == 32 ? 1 : 0, Pw, L.R, L.H, 1, 0,
                               PC_TRAIN_FWD, s, 0, 0, nullptr, fuse ? &st : nullptr));
      if (!fuse) {
        if (L.fmt == 32) tbn_stats_kernel<32><<<cap_grid(ctx, (vpix + 63) / 64 / 4 + 1, 2), 256, 0, s>>>(T.X[l], n, L.cout, L.H, Pw, L.pitch, sums);
        else tbn_stats_kernel<64><<<cap_grid(ctx, (vpix + 31) / 32 / 4 + 1, 2), 256, 0, s>>>(T.X[l], n, L.cout, L.H, Pw, L.pitch, sums);
        ctx->launches++;
      }
    }
    const double* cnt;
    SC_TRY(sync_sums(ctx, sums, (double)vpix, &cnt, s));
    // the activation kernels derive mean / inv-std from the sums themselves; their first CTA publishes them
    if (l < 4) {
      const int64_t opix = (int64_t)L.oR * n * L.oPitch;
      const unsigned grid = (unsigned)((opix + 63) / 64);
      if (L.fmt == 32)
        tbn_act_kernel<32><<<grid, 256, 0, s>>>(T.X[l], n, L.cout, Pw, L.pitch, sums, (double)vpix, cnt, T.mean[l], T.istd[l], G + Ob.bn[l][2], G + Ob.bn[l][3],
                                                P + Ob.bn[l][1], P + Ob.bn[l][0], P + Ob.alpha[l], L.pool, T.A[l], L.oR, L.oPitch, L.oH, T.idx[l], ctx->train_wgrad_mn ? nullptr : T.AT[l],
                                                pad8(L.cout));
      else
        tbn_act_kernel<64><<<grid, 512, 0, s>>>(T.X[l], n, L.cout, Pw, L.pitch, sums, (double)vpix, cnt, T.mean[l], T.istd[l], G + Ob.bn[l][2], G + Ob.bn[l][3],
                                                P + Ob.bn[l][1], P + Ob.bn[l][0], P + Ob.alpha[l], L.pool, T.A[l], L.oR, L.oPitch, L.oH, T.idx[l], ctx->train_wgrad_mn ? nullptr : T.AT[l],
                                                pad8(L.cout));
    } else {
      tact5_flatten_kernel<<<(unsigned)(((int64_t)n * 540 + 255) / 256), 256, 0, s>>>(T.X[4], n, sums, (double)vpix, cnt, T.mean[4], T.istd[4], G + Ob.bn[4][2],
                                                                                     G + Ob.bn[4][3], P + Ob.bn[4][1], P + Ob.bn[4][0], P + Ob.alpha[4],
                                                                                     masks + b * 540, F5);
    }
    ctx->launches++;
  }
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

template <int FMT, int DFMT>
static int bwd_layer(sc_ctx* ctx, int b, int l, const TcBranchBuf& T, const float* dA, const float* dF5, int dF5_ld, const uint8_t* mask, int n,
                     int dPw, int dPitch, float* frame, uint16_t* DT, float* planar, cudaStream_t s) {
  const TLayer& L = kTL[l];
  const BranchOff& Ob = ctx->off.br[b];
  float* P = ctx->params;
  float* G = ctx->grads;
  const int Pw = n * L.pitch;
  const int64_t vpix = (int64_t)L.H * n * L.H;
  constexpr int NCH = FMT / 8;
  double* sums = T.sums + (5 + l) * kSumsStride;
  tbn_bwd_reduce_kernel<FMT, DFMT><<<cap_grid(ctx, (vpix * NCH + 255) / 256 / 4 + 1, 2), 256, 0, s>>>(
      T.X[l], dA, T.idx[l], dF5, dF5_ld, mask, n, L.cout, L.H, Pw, L.pitch, L.pool, dPw, dPitch, T.mean[l], T.istd[l], P + Ob.bn[l][1], P + Ob.bn[l][0],
      P + Ob.alpha[l], sums);
  const bool hook = ctx->ar_hook != nullptr;     // synchronised BatchNorm: the LOCAL sums are the parameter gradients, copy them out before the all-reduce
  if (hook) { tbn_bwd_params_kernel<<<1, 64, 0, s>>>(sums, L.cout, G + Ob.bn[l][0], G + Ob.bn[l][1], G + Ob.alpha[l]); ctx->launches++; }
  const double* cnt;
  SC_TRY(sync_sums(ctx, sums, (double)vpix, &cnt, s));
  const int64_t npix = (int64_t)L.R * Pw;
  tbn_bwd_dx_kernel<FMT, DFMT><<<(unsigned)((npix + 63) / 64), 64 * NCH, 0, s>>>(
      T.X[l], dA, T.idx[l], dF5, dF5_ld, mask, n, L.cout, L.H, L.R, Pw, L.pitch, L.pool, dPw, dPitch, T.mean[l], T.istd[l], P + Ob.bn[l][1], P + Ob.bn[l][0],
      P + Ob.alpha[l], sums, (double)vpix, cnt, hook ? nullptr : G + Ob.bn[l][0], G + Ob.bn[l][1], G + Ob.alpha[l], frame, DT, pad8(L.cout), planar, 32);
  ctx->launches += 2;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// dF5: gradient of the flattened, dropped-out conv5 activation [n][540]
int tc_branch_backward(sc_ctx* ctx, int b, const TcBranchBuf& T, const float* patches, const float* dF5, int dF5_ld, const uint8_t* masks, int n,
                       cudaStream_t s) {
  const BranchOff& Ob = ctx->off.br[b];
  float* G = ctx->grads;
  uint16_t* DT = ctx->train_wgrad_mn ? nullptr : T.DT;     // the MN-major wgrad reads the frame itself: no planar gradient copies
  for (int l = 4; l >= 0; --l) {
    const TLayer& L = kTL[l];
    const int Pw = n * L.pitch;
    // the incoming gradient: conv5 <- dF5; pooled layers <- the dgrad output at the pooled geometry; others same geometry
    const int dPw = L.pool ? n * L.oPitch : Pw, dPitch = L.pool ? L.oPitch : L.pitch;
    if (l == 4) SC_TRY((bwd_layer<64, 64>(ctx, b, l, T, nullptr, dF5, dF5_ld, masks + b * 540, n, dPw, dPitch, T.frame, DT, nullptr, s)));
    else if (l == 3) SC_TRY((bwd_layer<64, 64>(ctx, b, l, T, T.dA, nullptr, 0, nullptr, n, dPw, dPitch, T.frame, DT, nullptr, s)));
    else if (l == 2) SC_TRY((bwd_layer<64, 64>(ctx, b, l, T, T.dA, nullptr, 0, nullptr, n, dPw, dPitch, T.frame, DT, nullptr, s)));
    else if (l == 1) SC_TRY((bwd_layer<32, 64>(ctx, b, l, T, T.dA, nullptr, 0, nullptr, n, dPw, dPitch, T.frame, DT, nullptr, s)));
    else {
      // conv1: reduction pass, then dx and the weight gradient in one fused pass (no dgrad below conv1)
      float* P = ctx->params;
      const int64_t vpix = (int64_t)30 * n * 30;
      double* sums = T.sums + 5 * kSumsStride;
      tbn_bwd_reduce_kernel<32, 32><<<cap_grid(ctx, (vpix * 4 + 255) / 256 / 4 + 1, 2), 256, 0, s>>>(
          T.X[0], T.dA, nullptr, nullptr, 0, nullptr, n, 20, 30, Pw, 32, 0, Pw, 32, T.mean[0], T.istd[0], P + Ob.bn[0][1], P + Ob.bn[0][0],
          P + Ob.alpha[0], sums);
      const bool hook = ctx->ar_hook != nullptr;
      if (hook) { tbn_bwd_params_kernel<<<1, 64, 0, s>>>(sums, 20, G + Ob.bn[0][0], G + Ob.bn[0][1], G + Ob.alpha[0]); ctx->launches++; }
      const double* cnt;
      SC_TRY(sync_sums(ctx, sums, (double)vpix, &cnt, s));
      ProfScope prof(ctx, PC_TRAIN_BWD, s);
      tbn_bwd_conv1_kernel<<<cap_grid(ctx, (vpix + 63) / 64 / 8 + 1, 2), 256, 0, s>>>(T.X[0], T.dA, patches, n, T.mean[0], T.istd[0], P + Ob.bn[0][1],
                                                                                    P + Ob.bn[0][0], P + Ob.alpha[0], sums, (double)vpix, cnt,
                                                                                    hook ? nullptr : G + Ob.bn[0][0], G + Ob.bn[0][1], G + Ob.alpha[0],
                                                                                    G + Ob.convW[0]);
      ctx->launches += 2;
      break;
    }
    const TLayer& Li = kTL[l - 1];
    const int64_t npix = (int64_t)L.R * Pw;
    if (ctx->train_wgrad_mn) SC_TRY(launch_wgrad_mn(ctx, T.A[l - 1], Li.fmt, T.frame, L.fmt, L.cin, L.cout, Pw, npix, L.H, G + Ob.convW[l], s));
    else SC_TRY(launch_wgrad_tc(ctx, T.AT[l - 1], T.DT, L.cin, L.cout, pad8(L.cin), pad16(L.cout), Pw, npix, L.H, G + Ob.convW[l], s));
    // dgrad: the gradient of this layer's input = sweep over the zero-framed dx with the raw taps; valid Li.oH x Li.oH
    SC_TRY(launch_conv_sweep(ctx, ctx->train_sw[b][l][1], l, T.frame, L.fmt == 32 ? 1 : 0, T.dA, (l == 1) ? 1 : 0, Pw, L.R, Li.oH, 1, 0,
                             PC_TRAIN_BWD, s, -2, -2));
  }
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
