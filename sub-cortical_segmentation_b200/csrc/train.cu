// Training step: nolearn's train_fn / eval_fn inside net.fit (cnn_cort/nets.py:233-246).
//
//   forward (training mode)  conv -> BatchNorm with BATCH statistics (biased variance, eps 1e-4) -> PReLU,
//                            pools after conv2 / conv4, dropout p=.5 (rescaled by 2) at *_l1drop, f1_drop, f2_drop,
//                            dense layers + PReLU, softmax, categorical cross-entropy (mean over the GLOBAL batch)
//   backward                 every parameter the reference trains: conv W, BN beta/gamma, PReLU alpha, dense W/b
//   output                   the context's flat gradient buffer (pickle layout).  The slots of the non-trainable BN
//                            running statistics carry this batch's mean / inv_std so that one all-reduce moves both;
//                            sc_adam_step applies Lasagne's Adam to the trainable entries and
//                            s <- 0.9 s + 0.1 batch (mean AND inv_std, Lasagne BatchNormLayer) to the statistics.
//
// BatchNorm's batch statistics force a grid-wide reduction between each conv and its activation, so the training
// forward is per-layer kernels.  The 3x3 convolutions (forward and dgrad) reuse the planar conv kernel of dense.cu
// with an identity epilogue; everything else is here.  All arithmetic fp32 FFMA; per-channel reductions accumulate
// in fp64 atomics.
#include "common.cuh"

namespace sc {

constexpr int kH[5] = {30, 28, 12, 10, 3};      // conv output size per layer
constexpr int kLd[5] = {32, 32, 16, 16, 8};     // row stride of the conv output maps
constexpr int kInH[5] = {32, 30, 14, 12, 5};    // conv input size
constexpr int kInLd[5] = {32, 32, 16, 16, 8};

// ---- parameter repacking ------------------------------------------------------------------------
// fwd: out[ci][t][co] = W[co][ci][8-t] (true convolution -> correlation taps);  dgrad: out[co][t][ci] = W[co][ci][t]
__global__ void repack_conv_kernel(const float* __restrict__ W, int cout, int cin, float* __restrict__ fwd, float* __restrict__ dgrad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * cin * 9) return;
  const int t = i % 9, ci = (i / 9) % cin, co = i / (9 * cin);
  const float v = W[i];
  fwd[(ci * 9 + (8 - t)) * cout + co] = v;
  if (dgrad) dgrad[(co * 9 + t) * cin + ci] = v;
}

// ---- BatchNorm statistics --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_stats_kernel(const float* __restrict__ x, int n, int C, int H, int W, int ld,
                                                       double* __restrict__ sums /*[C][2]*/) {
  const int c = blockIdx.x;
  const int64_t per = (int64_t)H * W, total = (int64_t)n * per;
  double s = 0.0, q = 0.0;
  for (int64_t e = (int64_t)blockIdx.y * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.y * 256) {
    const int i = (int)(e / per);
    const int r = (int)(e - (int64_t)i * per);
    const int h = r / W, w = r - h * W;
    const float v = x[(((int64_t)i * C + c) * H + h) * ld + w];
    s += v; q += (double)v * v;
  }
  for (int o = 16; o; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  __shared__ double ss[8], sq[8];
  if ((threadIdx.x & 31) == 0) { ss[threadIdx.x >> 5] = s; sq[threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { s += ss[w]; q += sq[w]; }
    atomicAdd(&sums[c * 2], s);
    atomicAdd(&sums[c * 2 + 1], q);
  }
}

__global__ void bn_finalize_kernel(const double* __restrict__ sums, int C, double count, float* __restrict__ mean,
                                   float* __restrict__ istd, float* __restrict__ g_mean_slot, float* __restrict__ g_istd_slot) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double m = sums[c * 2] / count;
  double var = sums[c * 2 + 1] / count - m * m;
  if (var < 0) var = 0;
  const float is = (float)(1.0 / sqrt(var + (double)kBnEps));
  mean[c] = (float)m; istd[c] = is;
  g_mean_slot[c] = (float)m; g_istd_slot[c] = is;   // carried to the optimiser through the gradient buffer
}

// y = (x-mean)*gamma*istd + beta; a = prelu(y); optional 2x2/2 max-pool with arg-max record
__global__ void bn_act_kernel(const float* __restrict__ x, int n, int C, int H, int W, int ld, const float* __restrict__ mean,
                              const float* __restrict__ istd, const float* __restrict__ gamma, const float* __restrict__ beta,
                              const float* __restrict__ alpha, int pool, float* __restrict__ out, int oH, int oW, int old,
                              uint8_t* __restrict__ idx) {
  const int64_t total = (int64_t)n * C * oH * oW;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(e % oW);
    const int h = (int)((e / oW) % oH);
    const int c = (int)((e / ((int64_t)oW * oH)) % C);
    const int i = (int)(e / ((int64_t)oW * oH * C));
    const float sc_ = gamma[c] * istd[c], sh = beta[c] - mean[c] * sc_, al = alpha[c];
    const float* xp = x + (((int64_t)i * C + c) * H) * ld;
    float r;
    if (!pool) {
      r = prelu(fmaf(xp[h * ld + w], sc_, sh), al);
    } else {
      int best = 0;
      r = prelu(fmaf(xp[(2 * h) * ld + 2 * w], sc_, sh), al);
#pragma unroll
      for (int k = 1; k < 4; ++k) {
        const float v = prelu(fmaf(xp[(2 * h + (k >> 1)) * ld + 2 * w + (k & 1)], sc_, sh), al);
        if (v > r) { r = v; best = k; }
      }
      idx[(((int64_t)i * C + c) * oH + h) * old + w] = (uint8_t)best;
    }
    out[(((int64_t)i * C + c) * oH + h) * old + w] = r;
  }
}

// ---- dropout ------------------------------------------------------------------------------------------
// mask layout per sample: [3][540] branch (c*9+h*3+w) | [540] f1_drop | [540] f2_drop
__global__ void make_masks_kernel(uint8_t* __restrict__ m, int64_t total, const unsigned long long* __restrict__ seed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) m[i] = (uint8_t)(hash3(*seed, (uint64_t)i) & 1u);   // the seed lives in device memory: the launch is graph-replayable
}

// conv5 activation [n][60][3][ld=8] -> F5 [n][540] with dropout
__global__ void flatten_drop_kernel(const float* __restrict__ a5, int n, const uint8_t* __restrict__ mask /*+b*540*/, float* __restrict__ f5) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)n * 540) return;
  const int i = (int)(e / 540), k = (int)(e - (int64_t)i * 540);
  const int c = k / 9, r = k - c * 9, h = r / 3, w = r - h * 3;
  const float v = a5[(((int64_t)i * 60 + c) * 3 + h) * 8 + w];
  f5[e] = mask[(int64_t)i * 2700 + k] ? 2.f * v : 0.f;
}
// d(F5) [n][540] -> d(A5) [n][60][3][8]
__global__ void unflatten_drop_kernel(const float* __restrict__ df5, int n, const uint8_t* __restrict__ mask, float* __restrict__ da5) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)n * 540) return;
  const int i = (int)(e / 540), k = (int)(e - (int64_t)i * 540);
  const int c = k / 9, r = k - c * 9, h = r / 3, w = r - h * 3;
  da5[(((int64_t)i * 60 + c) * 3 + h) * 8 + w] = mask[(int64_t)i * 2700 + k] ? 2.f * df5[e] : 0.f;
}

// ---- generic small SGEMM with guards: C[M][N] (+)= op(A)[M][K] * op(B)[K][N] ------------------------
// TA: A stored [K][M] (lda = M-stride);  TB: B stored [N][K].  beta0: overwrite, else accumulate (C += ...).
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb,
                                                    float* __restrict__ C, int ldc, int M, int N, int K,
                                                    const float* __restrict__ bias, int accumulate) {
  __shared__ float As[16][65], Bs[16][65];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int e = threadIdx.x; e < 1024; e += 256) {
      int kk, mm;
      if (TA) { mm = e & 63; kk = e >> 6; } else { kk = e & 15; mm = e >> 4; }
      const int gm = m0 + mm, gk = k0 + kk;
      As[kk][mm] = (gm < M && gk < K) ? (TA ? A[(int64_t)gk * lda + gm] : A[(int64_t)gm * lda + gk]) : 0.f;
      int nn;
      if (TB) { kk = e & 15; nn = e >> 4; } else { nn = e & 63; kk = e >> 6; }
      const int gn = n0 + nn; const int gk2 = k0 + kk;
      Bs[kk][nn] = (gn < N && gk2 < K) ? (TB ? B[(int64_t)gn * ldb + gk2] : B[(int64_t)gk2 * ldb + gn]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] + (bias ? bias[n] : 0.f);
      if (accumulate) v += C[(int64_t)m * ldc + n];
      C[(int64_t)m * ldc + n] = v;
    }
  }
}

template <bool TA, bool TB>
static int sgemm(sc_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int K,
                 const float* bias, int accumulate, int cls, cudaStream_t st) {
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  ProfScope prof(ctx, cls, st);
  sgemm_kernel<TA, TB><<<grid, 256, 0, st>>>(A, lda, B, ldb, C, ldc, M, N, K, bias, accumulate);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// dense PReLU forward: out[m][col0+j] = prelu(z[m][j], alpha[j]) * (mask ? 2*mask : 1)
__global__ void dense_act_kernel(const float* __restrict__ z, int M, int N, const float* __restrict__ alpha,
                                 const uint8_t* __restrict__ mask, int mask_ld, float* __restrict__ out, int out_ld, int col0) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)M * N) return;
  const int m = (int)(e / N), j = (int)(e - (int64_t)m * N);
  float v = prelu(z[e], alpha[j]);
  if (mask) v = mask[(int64_t)m * mask_ld + j] ? 2.f * v : 0.f;
  out[(int64_t)m * out_ld + col0 + j] = v;
}
// dense PReLU backward: dz = dy*(mask*2)*(z>0?1:alpha); galpha[j] += sum_m dyd*z*[z<=0]; gbias[j] += sum_m dz
__global__ void __launch_bounds__(256) dense_act_bwd_kernel(const float* __restrict__ dy, int dy_ld, int col0, const float* __restrict__ z,
                                                            int M, int N, const float* __restrict__ alpha, const uint8_t* __restrict__ mask,
                                                            int mask_ld, float* __restrict__ dz, float* __restrict__ galpha,
                                                            float* __restrict__ gbias) {
  const int j = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r0 = threadIdx.x >> 5;
  float sa = 0.f, sb = 0.f;
  if (j < N) {
    const float al = alpha[j];
    for (int m = blockIdx.y * 8 + r0; m < M; m += gridDim.y * 8) {
      float g = dy[(int64_t)m * dy_ld + col0 + j];
      if (mask) g = mask[(int64_t)m * mask_ld + j] ? 2.f * g : 0.f;
      const float zz = z[(int64_t)m * N + j];
      const float d = zz > 0.f ? g : al * g;
      dz[(int64_t)m * N + j] = d;
      if (zz <= 0.f) sa += g * zz;
      sb += d;
    }
  }
  __shared__ float ra[8][33], rb[8][33];
  ra[r0][threadIdx.x & 31] = sa; rb[r0][threadIdx.x & 31] = sb;
  __syncthreads();
  if (r0 == 0 && j < N) {
    for (int k = 1; k < 8; ++k) { sa += ra[k][threadIdx.x & 31]; sb += rb[k][threadIdx.x & 31]; }
    atomicAdd(&galpha[j], sa);
    atomicAdd(&gbias[j], sb);
  }
}
__global__ void colsum_kernel(const float* __restrict__ x, int M, int N, float* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  float s = 0.f;
  for (int m = blockIdx.y; m < M; m += gridDim.y) s += x[(int64_t)m * N + j];
  atomicAdd(&out[j], s);
}

// softmax + cross-entropy: dz = (p - onehot)/n_global, loss += sum(-log p[y])/n_global
__global__ void softmax_ce_kernel(const float* __restrict__ z, const uint8_t* __restrict__ y, int n, float inv_global,
                                  float* __restrict__ dz, float* __restrict__ loss) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.f;
  if (i < n) {
    float v[15], mx = -INFINITY, s = 0.f;
#pragma unroll
    for (int c = 0; c < 15; ++c) { v[c] = z[i * 15 + c]; mx = fmaxf(mx, v[c]); }
    const int t = y[i] < 15 ? y[i] : 0;   // raw label 15 (the boundary ring, base.py:89 maps it to 0) never indexes out of bounds
    const float zt = z[i * 15 + t] - mx;
#pragma unroll
    for (int c = 0; c < 15; ++c) { v[c] = expf(v[c] - mx); s += v[c]; }
    l = (logf(s) - zt) * inv_global;   // -log softmax[t], stable for saturated outputs
#pragma unroll
    for (int c = 0; c < 15; ++c) dz[i * 15 + c] = (v[c] / s - (c == t ? 1.f : 0.f)) * inv_global;
  }
  for (int o = 16; o; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  if ((threadIdx.x & 31) == 0 && l != 0.f) atomicAdd(loss, l);
}

// ---- conv block backward ------------------------------------------------------------------------------
// incoming gradient da: at pooled resolution (pool=1, routed through idx) or full resolution.
// pass 1: s[c] = {sum dy, sum dy*xhat, sum da*y*[y<=0]}   with y = xhat*gamma+beta, dy = da*(y>0?1:alpha)
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const float* __restrict__ x, const float* __restrict__ da, const uint8_t* __restrict__ idx,
                                                            int n, int C, int H, int W, int ld, int pool, int pld,
                                                            const float* __restrict__ mean, const float* __restrict__ istd,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            const float* __restrict__ alpha, double* __restrict__ sums /*[C][3]*/) {
  const int c = blockIdx.x;
  const int64_t per = (int64_t)H * W, total = (int64_t)n * per;
  const float mu = mean[c], is = istd[c], ga = gamma[c], be = beta[c], al = alpha[c];
  double s1 = 0, s2 = 0, s3 = 0;
  for (int64_t e = (int64_t)blockIdx.y * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.y * 256) {
    const int i = (int)(e / per);
    const int r = (int)(e - (int64_t)i * per);
    const int h = r / W, w = r - h * W;
    float g;
    if (pool) {
      const int64_t po = (((int64_t)i * C + c) * (H / 2) + (h >> 1)) * pld + (w >> 1);
      g = idx[po] == ((h & 1) * 2 + (w & 1)) ? da[po] : 0.f;
    } else {
      g = da[(((int64_t)i * C + c) * H + h) * ld + w];
    }
    const float xh = (x[(((int64_t)i * C + c) * H + h) * ld + w] - mu) * is;
    const float yv = fmaf(xh, ga, be);
    const float dy = yv > 0.f ? g : al * g;
    s1 += dy; s2 += (double)dy * xh;
    if (yv <= 0.f) s3 += (double)g * yv;
  }
  for (int o = 16; o; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); s3 += __shfl_xor_sync(0xffffffffu, s3, o);
  }
  __shared__ double sh[8][3];
  if ((threadIdx.x & 31) == 0) { sh[threadIdx.x >> 5][0] = s1; sh[threadIdx.x >> 5][1] = s2; sh[threadIdx.x >> 5][2] = s3; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { s1 += sh[w][0]; s2 += sh[w][1]; s3 += sh[w][2]; }
    atomicAdd(&sums[c * 3], s1); atomicAdd(&sums[c * 3 + 1], s2); atomicAdd(&sums[c * 3 + 2], s3);
  }
}
__global__ void bn_bwd_params_kernel(const double* __restrict__ sums, int C, float* __restrict__ gbeta, float* __restrict__ ggamma,
                                     float* __restrict__ galpha) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  gbeta[c] = (float)sums[c * 3]; ggamma[c] = (float)sums[c * 3 + 1]; galpha[c] = (float)sums[c * 3 + 2];
}
// pass 2: dx = gamma*istd*(dy - s1/m - xhat*s2/m), written (a) compact [n][C][H][ld] for wgrad and
// (b) zero-padded by 2 [n][C][H+4][pld2] for the dgrad convolution (borders pre-zeroed).
__global__ void bn_bwd_dx_kernel(const float* __restrict__ x, const float* __restrict__ da, const uint8_t* __restrict__ idx, int n, int C,
                                 int H, int W, int ld, int pool, int pld, const float* __restrict__ mean, const float* __restrict__ istd,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ alpha,
                                 const double* __restrict__ sums, double count, float* __restrict__ dx, float* __restrict__ dxpad, int pld2) {
  const int64_t total = (int64_t)n * C * H * W;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(e % W);
    const int h = (int)((e / W) % H);
    const int c = (int)((e / ((int64_t)W * H)) % C);
    const int i = (int)(e / ((int64_t)W * H * C));
    float g;
    if (pool) {
      const int64_t po = (((int64_t)i * C + c) * (H / 2) + (h >> 1)) * pld + (w >> 1);
      g = idx[po] == ((h & 1) * 2 + (w & 1)) ? da[po] : 0.f;
    } else {
      g = da[(((int64_t)i * C + c) * H + h) * ld + w];
    }
    const float is = istd[c], ga = gamma[c];
    const int64_t xo = (((int64_t)i * C + c) * H + h) * ld + w;
    const float xh = (x[xo] - mean[c]) * is;
    const float yv = fmaf(xh, ga, beta[c]);
    const float dy = yv > 0.f ? g : alpha[c] * g;
    const float r = ga * is * (dy - (float)(sums[c * 3] / count) - xh * (float)(sums[c * 3 + 1] / count));
    dx[xo] = r;
    if (dxpad) dxpad[(((int64_t)i * C + c) * (H + 4) + h + 2) * pld2 + w + 2] = r;
  }
}
// wgrad: gW[co][ci][ky][kx] = sum_{n,y,x} dx[n][co][y][x] * in[n][ci][y+2-ky][x+2-kx]
// one CTA per (co, ci, sample chunk); 9 taps per thread, block reduction, atomicAdd
__global__ void __launch_bounds__(128) conv_wgrad_kernel(const float* __restrict__ in, int Cin, int inH, int inLd, const float* __restrict__ dx,
                                                         int Cout, int H, int W, int ld, int n, float* __restrict__ gW) {
  const int co = blockIdx.x, ci = blockIdx.y;
  const int per = H * W;
  float acc[9] = {};
  for (int i = blockIdx.z; i < n; i += gridDim.z) {
    const float* dp = dx + ((int64_t)i * Cout + co) * H * ld;
    const float* ip = in + ((int64_t)i * Cin + ci) * inH * inLd;
    for (int e = threadIdx.x; e < per; e += 128) {
      const int y = e / W, xx = e - y * W;
      const float d = dp[y * ld + xx];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) acc[ky * 3 + kx] = fmaf(d, ip[(y + 2 - ky) * inLd + xx + 2 - kx], acc[ky * 3 + kx]);
    }
  }
  __shared__ float red[4][9];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    float v = acc[t];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][t] = v;
  }
  __syncthreads();
  if (threadIdx.x < 9) {
    const float v = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
    atomicAdd(&gW[((int64_t)co * Cin + ci) * 9 + threadIdx.x], v);
  }
}



// wgrad, register-tiled: one thread owns 4 output channels x 1 input channel x 9 taps (36 accumulators) and walks the
// pixels of its CTA's samples four at a time (sliding 6-wide input window per filter row: 22 shared loads per 144 FMA).
// CTA = (COUT/4) x 20 threads, one tile of 20 input channels, `spc` samples; one atomicAdd per accumulator at the end.
// PS row splits per CTA (threads = (COUT/4) x 20 x PS): split ps walks the output rows y = ps, ps + PS, ...; the partial sums
// are reduced through shared memory before the atomics.  Without the split a conv2 CTA has only 100 threads.
template <int COUT, int PS>
__global__ void __launch_bounds__((COUT / 4) * 20 * PS) conv_wgrad_tiled_kernel(const float* __restrict__ in, int Cin, int inH, int inLd,
                                                                               const float* __restrict__ dx, int H, int ld, int n, int spc,
                                                                               float* __restrict__ gW) {
  extern __shared__ __align__(16) float sm[];
  const int plane = (inH + 1) * inLd + 9;               // odd stride: the 20 channel planes fall into different banks
  const int planep = plane | 1;
  float* in_s = sm;                                      // [20][planep]
  float* dx_s = sm + ((20 * planep + 3) & ~3);           // [H*H][COUT]
  constexpr int NT1 = (COUT / 4) * 20;
  const int nthr = NT1 * PS;
  const int ps = threadIdx.x / NT1;
  const int tid = threadIdx.x, t1 = tid - ps * NT1, cog = t1 / 20, ci = t1 - cog * 20;
  const int ci0 = blockIdx.x * 20;
  const int s_begin = blockIdx.y * spc, s_end = min(n, s_begin + spc);
  float acc[4][9];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[c][t] = 0.f;
  for (int s = s_begin; s < s_end; ++s) {
    __syncthreads();
    for (int e = tid; e < 20 * planep; e += nthr) {
      const int c = e / planep, off = e - c * planep;
      const int r = off / inLd, col = off - r * inLd;
      float v = 0.f;
      if (r < inH && col < inH) v = __ldg(in + (((int64_t)s * Cin + ci0 + c) * inH + r) * inLd + col);
      in_s[e] = v;
    }
    for (int e = tid; e < COUT * H * H; e += nthr) {
      const int x = e % H, y = (e / H) % H, co = e / (H * H);
      dx_s[(y * H + x) * COUT + co] = __ldg(dx + (((int64_t)s * COUT + co) * H + y) * ld + x);
    }
    __syncthreads();
    const float* ip = in_s + ci * planep;
    for (int y = ps; y < H; y += PS) {
      for (int x0 = 0; x0 < H; x0 += 4) {
        float d[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (x0 + j < H) v = *reinterpret_cast<const float4*>(dx_s + (y * H + x0 + j) * COUT + cog * 4);
          d[j][0] = v.x; d[j][1] = v.y; d[j][2] = v.z; d[j][3] = v.w;
        }
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
          float row[6];
          const float* rp = ip + (y + 2 - ky) * inLd + x0;
#pragma unroll
          for (int k = 0; k < 6; ++k) row[k] = rp[k];
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int c = 0; c < 4; ++c) acc[c][ky * 3 + kx] = fmaf(d[j][c], row[j + 2 - kx], acc[c][ky * 3 + kx]);
        }
      }
    }
  }
  if (PS > 1) {   // reduce the row splits through shared memory (the staging buffers are free now)
    __syncthreads();
    float* red = sm;                                       // [PS - 1][36][NT1]
    if (ps > 0) {
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int t = 0; t < 9; ++t) red[((ps - 1) * 36 + c * 9 + t) * NT1 + t1] = acc[c][t];
    }
    __syncthreads();
    if (ps > 0) return;
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int t = 0; t < 9; ++t)
        for (int q = 0; q < PS - 1; ++q) acc[c][t] += red[(q * 36 + c * 9 + t) * NT1 + t1];
  }
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int t = 0; t < 9; ++t) atomicAdd(&gW[((int64_t)(cog * 4 + c) * Cin + ci0 + ci) * 9 + t], acc[c][t]);
}

template <int COUT>
static int launch_wgrad_tiled(sc_ctx* ctx, const float* in, int Cin, int inH, int inLd, const float* dx, int H, int ld, int n,
                              float* gW, cudaStream_t st) {
  constexpr int PS = COUT == 20 ? 4 : (COUT == 40 ? 2 : 1);     // ~400 threads per CTA
  const int planep = ((inH + 1) * inLd + 9) | 1;
  size_t smem_f = (size_t)((20 * planep + 3) & ~3) + (size_t)COUT * H * H;
  const size_t red_f = (size_t)(PS - 1) * 36 * (COUT / 4) * 20;
  if (PS > 1 && smem_f < red_f) smem_f = red_f;
  const size_t smem = smem_f * sizeof(float);
  auto kern = conv_wgrad_tiled_kernel<COUT, PS>;
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), (int)smem));
  // samples per CTA: ~2 000 pixels of reduction each, but never fewer than ~2 CTAs per SM
  int spc = 2048 / (H * H);
  const int fill = (n * (Cin / 20) + 2 * ctx->sm_count - 1) / (2 * ctx->sm_count);
  if (spc > fill) spc = fill;
  if (spc < 1) spc = 1;
  dim3 grid(Cin / 20, (n + spc - 1) / spc);
  ProfScope prof(ctx, PC_TRAIN_BWD, st);
  kern<<<grid, (COUT / 4) * 20 * PS, smem, st>>>(in, Cin, inH, inLd, dx, H, ld, n, spc, gW);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---- 3x3 valid convolution over small planar maps (training forward and dgrad) ----------------------------------
// Same register tiling as the dense-path conv kernel (320 threads = 64 pixel groups of 8 columns x 5 channel groups,
// input channels staged through shared memory in chunks of 10), but the 64 pixel groups are spread over
// NS samples x TH rows x SEG column segments so that the 3x3 .. 30x30 training maps do not waste a 16x32 tile.
template <int CIN, int COUT, int NS, int TH, int SEG>
struct TConvCfg {
  static constexpr int CHUNK = 10, CO_T = COUT / 5;
  static constexpr int IH = TH + 2, IW = SEG * 8 + 4, IWP = IW;   // IW == 4 (mod 8): conflict-free LDS.128
  static constexpr int IN_FLOATS = CHUNK * NS * IH * IWP, W_FLOATS = CHUNK * 9 * COUT;
  static constexpr size_t SMEM = (size_t)(IN_FLOATS + W_FLOATS) * sizeof(float);
  static_assert(NS * TH * SEG == 64, "64 pixel groups per CTA");
};

template <int CIN, int COUT, int NS, int TH, int SEG>
__global__ void __launch_bounds__(320) train_conv_kernel(const float* __restrict__ in, int inR, int inLd, float* __restrict__ out,
                                                         int outR, int outLd, const float* __restrict__ w, int n) {
  using Cfg = TConvCfg<CIN, COUT, NS, TH, SEG>;
  extern __shared__ __align__(16) float smem[];
  float* s_in = smem;
  float* s_w = smem + Cfg::IN_FLOATS;
  const int tid = threadIdx.x;
  const int cg = tid >> 6, pg = tid & 63;
  const int seg = pg % SEG, prow = (pg / SEG) % TH, smp = pg / (SEG * TH);
  const int tr0 = blockIdx.y * TH, tc0 = blockIdx.x * SEG * 8, s0 = blockIdx.z * NS;
  float acc[8][Cfg::CO_T];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int c = 0; c < Cfg::CO_T; ++c) acc[p][c] = 0.f;
  for (int ci0 = 0; ci0 < CIN; ci0 += Cfg::CHUNK) {
    __syncthreads();
    for (int e = tid; e < Cfg::CHUNK * NS * Cfg::IH * Cfg::IW; e += 320) {
      const int col = e % Cfg::IW;
      const int row = (e / Cfg::IW) % Cfg::IH;
      const int sm = (e / (Cfg::IW * Cfg::IH)) % NS;
      const int ci = e / (Cfg::IW * Cfg::IH * NS);
      const int gr = tr0 + row, gc = tc0 + col, gs = s0 + sm;
      float v = 0.f;
      if (gs < n && gr < inR && gc < inLd) v = __ldg(in + (((int64_t)gs * CIN + ci0 + ci) * inR + gr) * inLd + gc);
      s_in[((ci * NS + sm) * Cfg::IH + row) * Cfg::IWP + col] = v;
    }
    for (int e = tid; e < Cfg::W_FLOATS / 4; e += 320)
      reinterpret_cast<float4*>(s_w)[e] = __ldg(reinterpret_cast<const float4*>(w + (int64_t)ci0 * 9 * COUT) + e);
    __syncthreads();
#pragma unroll 1
    for (int ci = 0; ci < Cfg::CHUNK; ++ci) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        float x[12];
        const float4* src = reinterpret_cast<const float4*>(s_in + ((ci * NS + smp) * Cfg::IH + prow + ky) * Cfg::IWP + seg * 8);
#pragma unroll
        for (int v = 0; v < 3; ++v) { const float4 t = src[v]; x[v * 4] = t.x; x[v * 4 + 1] = t.y; x[v * 4 + 2] = t.z; x[v * 4 + 3] = t.w; }
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          float wv[Cfg::CO_T];
          const float4* wsrc = reinterpret_cast<const float4*>(s_w + (ci * 9 + ky * 3 + kx) * COUT + cg * Cfg::CO_T);
#pragma unroll
          for (int v = 0; v < Cfg::CO_T / 4; ++v) { const float4 t = wsrc[v]; wv[v * 4] = t.x; wv[v * 4 + 1] = t.y; wv[v * 4 + 2] = t.z; wv[v * 4 + 3] = t.w; }
#pragma unroll
          for (int p = 0; p < 8; ++p)
#pragma unroll
            for (int c = 0; c < Cfg::CO_T; ++c) acc[p][c] = fmaf(x[kx + p], wv[c], acc[p][c]);
        }
      }
    }
  }
  const int orow = tr0 + prow, ocol = tc0 + seg * 8, os = s0 + smp;
  if (os >= n || orow >= outR || ocol >= outLd) return;
#pragma unroll
  for (int c = 0; c < Cfg::CO_T; ++c) {
    float* o = out + (((int64_t)os * COUT + cg * Cfg::CO_T + c) * outR + orow) * outLd + ocol;
    *reinterpret_cast<float4*>(o) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[3][c]);
    *reinterpret_cast<float4*>(o + 4) = make_float4(acc[4][c], acc[5][c], acc[6][c], acc[7][c]);
  }
}

template <int CIN, int COUT, int NS, int TH, int SEG>
static int launch_tconv(sc_ctx* ctx, const float* in, int inR, int inLd, float* out, int outR, int outLd, const float* w, int n,
                        int cls, cudaStream_t st) {
  using Cfg = TConvCfg<CIN, COUT, NS, TH, SEG>;
  auto kern = train_conv_kernel<CIN, COUT, NS, TH, SEG>;
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), (int)Cfg::SMEM));
  dim3 grid((outLd + SEG * 8 - 1) / (SEG * 8), (outR + TH - 1) / TH, (n + NS - 1) / NS);
  ProfScope prof(ctx, cls, st);
  kern<<<grid, 320, Cfg::SMEM, st>>>(in, inR, inLd, out, outR, outLd, w, n);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// dispatch by (cin, cout, output size): forward conv2..conv5 and the four dgrads
static int train_conv(sc_ctx* ctx, int cin, int cout, const float* in, int inR, int inLd, float* out, int outR, int outLd,
                      const float* w, int n, int cls, cudaStream_t st) {
  if (cin == 20 && cout == 20) return launch_tconv<20, 20, 1, 16, 4>(ctx, in, inR, inLd, out, outR, outLd, w, n, cls, st);
  if (cin == 20 && cout == 40) return launch_tconv<20, 40, 2, 16, 2>(ctx, in, inR, inLd, out, outR, outLd, w, n, cls, st);
  if (cin == 40 && cout == 40) return launch_tconv<40, 40, 2, 16, 2>(ctx, in, inR, inLd, out, outR, outLd, w, n, cls, st);
  if (cin == 40 && cout == 60) return launch_tconv<40, 60, 16, 4, 1>(ctx, in, inR, inLd, out, outR, outLd, w, n, cls, st);
  if (cin == 60 && cout == 40) return launch_tconv<60, 40, 8, 8, 1>(ctx, in, inR, inLd, out, outR, outLd, w, n, cls, st);
  if (cin == 40 && cout == 20) return launch_tconv<40, 20, 2, 16, 2>(ctx, in, inR, inLd, out, outR, outLd, w, n, cls, st);
  set_error("train_conv: unsupported channel pair %d -> %d", cin, cout);
  return SC_ERR_ARG;
}

// ---- optimiser -------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            const uint8_t* __restrict__ trainable, int n, float a_t, float b1, float b2, float eps, float gscale,
                            float sscale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t t = trainable[i];
  if (t == 1) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] = p[i] - a_t * mi / (sqrtf(vi) + eps);
  } else if (t == 0) {
    p[i] = 0.9f * p[i] + 0.1f * (g[i] * sscale);   // BN running mean / inv_std (Lasagne alpha = 0.1)
  }                                                 // 2: frozen (sc_freeze_trunk), parameter and moments untouched
}

int adam_step(sc_ctx* ctx, float lr, float b1, float b2, float eps, float gscale, float sscale, cudaStream_t st) {
  ctx->adam_t += 1;
  const double t = (double)ctx->adam_t;
  const float a_t = (float)(lr * sqrt(1.0 - pow((double)b2, t)) / (1.0 - pow((double)b1, t)));
  ProfScope prof(ctx, PC_ADAM, st);
  adam_kernel<<<(SC_PARAM_FLOATS + 255) / 256, 256, 0, st>>>(ctx->params, ctx->grads, ctx->adam_m, ctx->adam_v, ctx->trainable,
                                                             SC_PARAM_FLOATS, a_t, b1, b2, eps, gscale, sscale);
  ctx->launches++;
  ctx->derived_dirty = true;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---- the step ------------------------------------------------------------------------------------------------
struct Bump {
  char* base; size_t off;
  template <class T> T* take(size_t count) {
    T* p = reinterpret_cast<T*>(base + off);
    off += (count * sizeof(T) + 255) & ~(size_t)255;
    return p;
  }
};

static unsigned ew_grid(int64_t total) { return (unsigned)((total + 255) / 256 < 65535 * 8 ? (total + 255) / 256 : 65535 * 8); }

// ---- the step buffers: the staged batch, then the selected back-end's buffers
struct SimtBuf {       // the exact-fp32 SIMT back-end (gemm = 0): planar fp32 maps and plain dense activations
  struct Branch {
    float* X[5]; float* A[5]; uint8_t* idx[2]; float* mean[5]; float* istd[5];
    float* F5; float* Z1;
    float* wf[5]; float* wd[5];
    float *dZ1, *dF5, *dA, *dX, *dXpad;
    double* sums;
  } bb[3];
  float *CAT, *ZF1, *CAT2, *ZF2, *H2, *ZO, *dZO, *dH2, *dZF2, *dCAT2, *dZF1, *dCAT;
};
struct StepBuf {
  float *in[3], *in4; uint8_t* y;      // the caller's batch, staged (the head-only step: in4 / y gathered from its tables)
  uint8_t* masks;
  unsigned long long* seed;
  float* loss;
  int64_t* idx;                        // head-only step: the staged row indices (unused without an index list)
  const HeadGather* head = nullptr;    // head-only step of fine-tuning: gather of cached trunk features, no convolutions
  SimtBuf simt;                        // gemm = 0
  TcBranchBuf tc[3];                   // gemm = 1
  TcDenseBuf td;
};

static void carve_simt(SimtBuf& M, Bump& B, int n) {
  for (int b = 0; b < 3; ++b) {
    auto& bb = M.bb[b];
    for (int l = 0; l < 5; ++l) {
      bb.X[l] = B.take<float>((size_t)n * kConvCout[l] * kH[l] * kLd[l]);
      const int oh = (l == 1 || l == 3) ? kH[l] / 2 : kH[l];
      const int old = (l == 1) ? 16 : (l == 3) ? 8 : kLd[l];
      bb.A[l] = B.take<float>((size_t)n * kConvCout[l] * oh * old);
      bb.mean[l] = B.take<float>(64); bb.istd[l] = B.take<float>(64);
      bb.wf[l] = B.take<float>((size_t)kConvCout[l] * kConvCin[l] * 9);
      bb.wd[l] = l > 0 ? B.take<float>((size_t)kConvCout[l] * kConvCin[l] * 9) : nullptr;
    }
    bb.idx[0] = B.take<uint8_t>((size_t)n * 20 * 14 * 16);
    bb.idx[1] = B.take<uint8_t>((size_t)n * 40 * 5 * 8);
    bb.F5 = B.take<float>((size_t)n * 540);
    bb.Z1 = B.take<float>((size_t)n * 180);
    bb.dZ1 = B.take<float>((size_t)n * 180);
    bb.dF5 = B.take<float>((size_t)n * 540);
    bb.dA = B.take<float>((size_t)n * 20 * 30 * 32);      // incoming activation gradient of the current layer
    bb.dX = B.take<float>((size_t)n * 20 * 30 * 32);      // compact conv-output gradient
    bb.dXpad = B.take<float>((size_t)n * 20 * 34 * 32);   // zero-padded copy for dgrad
    bb.sums = B.take<double>(64 * 3);
  }
  M.CAT = B.take<float>((size_t)n * 540);     // [D1_ax | D1_cor | D1_sag], f1_drop applied
  M.ZF1 = B.take<float>((size_t)n * 540);
  M.CAT2 = B.take<float>((size_t)n * 555);    // [prelu(ZF1) with f2_drop | atlas]
  M.ZF2 = B.take<float>((size_t)n * 270);
  M.H2 = B.take<float>((size_t)n * 270);
  M.ZO = B.take<float>((size_t)n * 15);
  M.dZO = B.take<float>((size_t)n * 15);
  M.dH2 = B.take<float>((size_t)n * 270);
  M.dZF2 = B.take<float>((size_t)n * 270);
  M.dCAT2 = B.take<float>((size_t)n * 555);
  M.dZF1 = B.take<float>((size_t)n * 540);
  M.dCAT = B.take<float>((size_t)n * 540);
}

// head: the head-only step (tensor cores only) keeps no patches and no conv maps
static size_t carve_step(StepBuf& S, char* base, int n, bool tc, bool head = false) {
  Bump B{base, 0};
  if (!head)
    for (int b = 0; b < 3; ++b) S.in[b] = B.take<float>((size_t)n * 1024);
  S.in4 = B.take<float>((size_t)n * 15);
  S.y = B.take<uint8_t>((size_t)n);
  S.masks = B.take<uint8_t>((size_t)n * 2700);
  S.seed = B.take<unsigned long long>(1);
  S.loss = B.take<float>(1);
  if (head) S.idx = B.take<int64_t>((size_t)n);
  if (tc) {
    if (!head)
      for (int b = 0; b < 3; ++b) tc_carve_branch(S.tc[b], B.take<char>(tc_branch_bytes(n)), n);
    tdense_carve(S.td, B.take<char>(tdense_bytes(n)), n);
  } else {
    carve_simt(S.simt, B, n);
  }
  return B.off;
}

// ---- SIMT back-end: conv1..conv5 with BatchNorm / PReLU / pools, d1 into CAT
static int simt_branch_forward(sc_ctx* ctx, int b, const StepBuf& S, int n, cudaStream_t s) {
  const BranchOff& Ob = ctx->off.br[b];
  const auto& bb = S.simt.bb[b];
  float* P = ctx->params;
  float* G = ctx->grads;
  const float* ones = ctx->train_consts;
  const float* zeros = ctx->train_consts + kTrainZeros;
  for (int l = 0; l < 5; ++l) {
    const int co = kConvCout[l], ci = kConvCin[l];
    repack_conv_kernel<<<(co * ci * 9 + 255) / 256, 256, 0, s>>>(P + Ob.convW[l], co, ci, bb.wf[l], bb.wd[l]);
    ctx->launches++;
    if (l == 0) {
      SC_TRY(launch_conv1_patches(ctx, S.in[b], n, bb.wf[0], ones, zeros, ones, bb.X[0], s));
    } else {
      SC_TRY(train_conv(ctx, ci, co, bb.A[l - 1], kInH[l], kInLd[l], bb.X[l], kH[l], kLd[l], bb.wf[l], n, PC_TRAIN_FWD, s));
    }
    SC_CUDA(cudaMemsetAsync(bb.sums, 0, 64 * 3 * sizeof(double), s));
    bn_stats_kernel<<<dim3(co, 32), 256, 0, s>>>(bb.X[l], n, co, kH[l], kH[l], kLd[l], bb.sums);
    bn_finalize_kernel<<<1, 64, 0, s>>>(bb.sums, co, (double)n * kH[l] * kH[l], bb.mean[l], bb.istd[l], G + Ob.bn[l][2], G + Ob.bn[l][3]);
    const int pool = (l == 1 || l == 3);
    const int oh = pool ? kH[l] / 2 : kH[l];
    const int old = (l == 1) ? 16 : (l == 3) ? 8 : kLd[l];
    bn_act_kernel<<<ew_grid((int64_t)n * co * oh * oh), 256, 0, s>>>(bb.X[l], n, co, kH[l], kH[l], kLd[l], bb.mean[l], bb.istd[l],
                                                                   P + Ob.bn[l][1], P + Ob.bn[l][0], P + Ob.alpha[l], pool, bb.A[l], oh, oh, old,
                                                                   pool ? bb.idx[l == 1 ? 0 : 1] : nullptr);
    ctx->launches += 3;
  }
  flatten_drop_kernel<<<ew_grid((int64_t)n * 540), 256, 0, s>>>(bb.A[4], n, S.masks + b * 540, bb.F5);
  SC_TRY((sgemm<false, false>(ctx, bb.F5, 540, P + Ob.d1W, 180, bb.Z1, 180, n, 180, 540, P + Ob.d1b, 0, PC_TRAIN_FWD, s)));
  dense_act_kernel<<<ew_grid((int64_t)n * 180), 256, 0, s>>>(bb.Z1, n, 180, P + Ob.d1alpha, S.masks + 1620 + b * 180, 2700, S.simt.CAT, 540, b * 180);
  ctx->launches += 2;
  return SC_OK;
}

// FC1 -> fc_2 -> out_layer -> softmax cross-entropy, then the backward pass of the head down to dCAT
static int simt_head(sc_ctx* ctx, const StepBuf& S, int n, int64_t n_global, cudaStream_t st) {
  const ParamOff& O = ctx->off;
  const SimtBuf& M = S.simt;
  float* P = ctx->params;
  float* G = ctx->grads;
  SC_TRY((sgemm<false, false>(ctx, M.CAT, 540, P + O.fc1W, 540, M.ZF1, 540, n, 540, 540, P + O.fc1b, 0, PC_TRAIN_FWD, st)));
  dense_act_kernel<<<ew_grid((int64_t)n * 540), 256, 0, st>>>(M.ZF1, n, 540, P + O.a1, S.masks + 2160, 2700, M.CAT2, 555, 0);
  SC_CUDA(cudaMemcpy2DAsync(M.CAT2 + 540, 555 * 4, S.in4, 15 * 4, 15 * 4, n, cudaMemcpyDeviceToDevice, st));
  SC_TRY((sgemm<false, false>(ctx, M.CAT2, 555, P + O.fc2W, 270, M.ZF2, 270, n, 270, 555, P + O.fc2b, 0, PC_TRAIN_FWD, st)));
  dense_act_kernel<<<ew_grid((int64_t)n * 270), 256, 0, st>>>(M.ZF2, n, 270, P + O.a2, nullptr, 0, M.H2, 270, 0);
  SC_TRY((sgemm<false, false>(ctx, M.H2, 270, P + O.outW, 15, M.ZO, 15, n, 15, 270, P + O.outb, 0, PC_TRAIN_FWD, st)));
  softmax_ce_kernel<<<(n + 127) / 128, 128, 0, st>>>(M.ZO, S.y, n, 1.f / (float)n_global, M.dZO, S.loss);
  ctx->launches += 3;
  // out layer
  SC_TRY((sgemm<true, false>(ctx, M.H2, 270, M.dZO, 15, G + O.outW, 15, 270, 15, n, nullptr, 0, PC_TRAIN_BWD, st)));
  colsum_kernel<<<dim3(1, 32), 32, 0, st>>>(M.dZO, n, 15, G + O.outb);
  SC_TRY((sgemm<false, true>(ctx, M.dZO, 15, P + O.outW, 15, M.dH2, 270, n, 270, 15, nullptr, 0, PC_TRAIN_BWD, st)));
  // fc_2
  dense_act_bwd_kernel<<<dim3((270 + 31) / 32, 16), 256, 0, st>>>(M.dH2, 270, 0, M.ZF2, n, 270, P + O.a2, nullptr, 0, M.dZF2, G + O.a2, G + O.fc2b);
  SC_TRY((sgemm<true, false>(ctx, M.CAT2, 555, M.dZF2, 270, G + O.fc2W, 270, 555, 270, n, nullptr, 0, PC_TRAIN_BWD, st)));
  SC_TRY((sgemm<false, true>(ctx, M.dZF2, 270, P + O.fc2W, 270, M.dCAT2, 555, n, 555, 270, nullptr, 0, PC_TRAIN_BWD, st)));
  // FC1 (dropout f2_drop sits on its activation)
  dense_act_bwd_kernel<<<dim3((540 + 31) / 32, 16), 256, 0, st>>>(M.dCAT2, 555, 0, M.ZF1, n, 540, P + O.a1, S.masks + 2160, 2700, M.dZF1, G + O.a1, G + O.fc1b);
  SC_TRY((sgemm<true, false>(ctx, M.CAT, 540, M.dZF1, 540, G + O.fc1W, 540, 540, 540, n, nullptr, 0, PC_TRAIN_BWD, st)));
  SC_TRY((sgemm<false, true>(ctx, M.dZF1, 540, P + O.fc1W, 540, M.dCAT, 540, n, 540, 540, nullptr, 0, PC_TRAIN_BWD, st)));
  ctx->launches += 3;
  return SC_OK;
}

// d1 (dropout f1_drop sits on the concatenated d1 activations), then conv5..conv1
static int simt_branch_backward(sc_ctx* ctx, int b, const StepBuf& S, int n, cudaStream_t s) {
  const BranchOff& Ob = ctx->off.br[b];
  const auto& bb = S.simt.bb[b];
  float* P = ctx->params;
  float* G = ctx->grads;
  dense_act_bwd_kernel<<<dim3((180 + 31) / 32, 16), 256, 0, s>>>(S.simt.dCAT, 540, b * 180, bb.Z1, n, 180, P + Ob.d1alpha, S.masks + 1620 + b * 180, 2700,
                                                                bb.dZ1, G + Ob.d1alpha, G + Ob.d1b);
  SC_TRY((sgemm<true, false>(ctx, bb.F5, 540, bb.dZ1, 180, G + Ob.d1W, 180, 540, 180, n, nullptr, 0, PC_TRAIN_BWD, s)));
  SC_TRY((sgemm<false, true>(ctx, bb.dZ1, 180, P + Ob.d1W, 180, bb.dF5, 540, n, 540, 180, nullptr, 0, PC_TRAIN_BWD, s)));
  ctx->launches++;
  unflatten_drop_kernel<<<ew_grid((int64_t)n * 540), 256, 0, s>>>(bb.dF5, n, S.masks + b * 540, bb.dA);
  ctx->launches++;
  for (int l = 4; l >= 0; --l) {
    const int co = kConvCout[l], ci = kConvCin[l], H = kH[l], ld = kLd[l];
    const int pool = (l == 1 || l == 3);
    const int pld = (l == 1) ? 16 : 8;
    const uint8_t* idx = pool ? bb.idx[l == 1 ? 0 : 1] : nullptr;
    const double count = (double)n * H * H;
    SC_CUDA(cudaMemsetAsync(bb.sums, 0, 64 * 3 * sizeof(double), s));
    bn_bwd_reduce_kernel<<<dim3(co, 32), 256, 0, s>>>(bb.X[l], bb.dA, idx, n, co, H, H, ld, pool, pld, bb.mean[l], bb.istd[l],
                                                      P + Ob.bn[l][1], P + Ob.bn[l][0], P + Ob.alpha[l], bb.sums);
    bn_bwd_params_kernel<<<1, 64, 0, s>>>(bb.sums, co, G + Ob.bn[l][0], G + Ob.bn[l][1], G + Ob.alpha[l]);
    const int pld2 = kInLd[l];   // padded map has the size of this layer's input (H+4 >= inH, same row stride)
    if (l > 0) SC_CUDA(cudaMemsetAsync(bb.dXpad, 0, (size_t)n * co * (H + 4) * pld2 * 4, s));
    bn_bwd_dx_kernel<<<ew_grid((int64_t)n * co * H * H), 256, 0, s>>>(bb.X[l], bb.dA, idx, n, co, H, H, ld, pool, pld, bb.mean[l], bb.istd[l],
                                                                     P + Ob.bn[l][1], P + Ob.bn[l][0], P + Ob.alpha[l], bb.sums, count, bb.dX,
                                                                     l > 0 ? bb.dXpad : nullptr, pld2);
    // wgrad against this layer's input (the previous activation, or the patches for conv1)
    const float* lin = l == 0 ? S.in[b] : bb.A[l - 1];
    if (l == 0) {
      int zc = n < 32 ? n : 32;
      conv_wgrad_kernel<<<dim3(co, ci, zc), 128, 0, s>>>(lin, ci, kInH[l], kInLd[l], bb.dX, co, H, H, ld, n, G + Ob.convW[l]);
      ctx->launches++;
    } else if (co == 20) {
      SC_TRY(launch_wgrad_tiled<20>(ctx, lin, ci, kInH[l], kInLd[l], bb.dX, H, ld, n, G + Ob.convW[l], s));
    } else if (co == 40) {
      SC_TRY(launch_wgrad_tiled<40>(ctx, lin, ci, kInH[l], kInLd[l], bb.dX, H, ld, n, G + Ob.convW[l], s));
    } else {
      SC_TRY(launch_wgrad_tiled<60>(ctx, lin, ci, kInH[l], kInLd[l], bb.dX, H, ld, n, G + Ob.convW[l], s));
    }
    ctx->launches += 3;
    if (l > 0) {
      // dgrad: d(input) = valid conv of the zero-padded dx with the raw taps, channel roles swapped
      SC_TRY(train_conv(ctx, co, ci, bb.dXpad, H + 4, pld2, bb.dA, kInH[l], kInLd[l], bb.wd[l], n, PC_TRAIN_BWD, s));
    }
  }
  return SC_OK;
}

// ---- tcgen05 back-end: the split-bf16 conv maps of train_tc.cu and the dense layers of train_dense.cu
static int tcgen05_branch_forward(sc_ctx* ctx, int b, const StepBuf& S, int n, cudaStream_t s) {
  const TcBranchBuf& T = S.tc[b];
  repack_conv_kernel<<<1, 256, 0, s>>>(ctx->params + ctx->off.br[b].convW[0], 20, 1, T.wf0, nullptr);
  ctx->launches++;
  SC_TRY(tc_branch_forward(ctx, b, T, S.in[b], n, S.masks, s));
  return tdense_branch_forward(ctx, b, S.td, T.F5, n, S.masks, s);
}

static int tcgen05_branch_backward(sc_ctx* ctx, int b, const StepBuf& S, int n, cudaStream_t s) {
  SC_TRY(tdense_branch_backward(ctx, b, S.td, n, S.masks, true, s));
  return tc_branch_backward(ctx, b, S.tc[b], S.in[b], S.td.dF5[b], 576, S.masks, n, s);
}

// The step body.  Every pointer it touches lives in the context (staged inputs, arena, parameter / gradient buffers), every
// scalar that changes from step to step is read from device memory (the dropout seed), so the same sequence of launches is
// valid as a captured CUDA graph.  The three branches are independent between the patches and the concatenation (forward)
// and after the gradient of the concatenation (backward): they run on three streams forked from / joined into `st`.
// With S.head (fine-tuning) the branches start at d1: one gather writes d1's operands from the cached trunk features, and
// the backward pass stops at d1's weight gradients.  Every trunk entry of the gradient buffer then stays 0.
static int train_body(sc_ctx* ctx, const StepBuf& S, int n, int64_t n_global, bool injected_masks, cudaStream_t st) {
  const bool tc = ctx->gemm_backend == 1;
  cudaStream_t sb[3] = {st, ctx->train_side[0], ctx->train_side[1]};
  cudaEvent_t* ev = ctx->train_ev;

  SC_CUDA(cudaMemsetAsync(ctx->grads, 0, sizeof(float) * SC_PARAM_FLOATS, st));
  SC_CUDA(cudaMemsetAsync(S.loss, 0, sizeof(float), st));
  if (!injected_masks) { make_masks_kernel<<<ew_grid((int64_t)n * 2700), 256, 0, st>>>(S.masks, (int64_t)n * 2700, S.seed); ctx->launches++; }
  if (S.head) SC_TRY(launch_head_gather(ctx, *S.head, st));
  SC_CUDA(cudaEventRecord(ev[0], st));
  for (int b = 1; b < 3; ++b) SC_CUDA(cudaStreamWaitEvent(sb[b], ev[0], 0));

  // forward of the branches, then the head (forward and backward) on `st`
  for (int b = 0; b < 3; ++b) {
    if (S.head) SC_TRY(tdense_branch_forward(ctx, b, S.td, nullptr, n, S.masks, sb[b]));
    else SC_TRY(tc ? tcgen05_branch_forward(ctx, b, S, n, sb[b]) : simt_branch_forward(ctx, b, S, n, sb[b]));
    if (b > 0) { SC_CUDA(cudaEventRecord(ev[b], sb[b])); SC_CUDA(cudaStreamWaitEvent(st, ev[b], 0)); }
  }
  SC_TRY(tc ? tdense_head(ctx, S.td, S.in4, S.y, n, n_global, S.masks, S.loss, st) : simt_head(ctx, S, n, n_global, st));
  SC_CUDA(cudaEventRecord(ev[3], st));
  for (int b = 1; b < 3; ++b) SC_CUDA(cudaStreamWaitEvent(sb[b], ev[3], 0));

  // backward of the branches
  for (int b = 0; b < 3; ++b) {
    if (S.head) SC_TRY(tdense_branch_backward(ctx, b, S.td, n, S.masks, false, sb[b]));
    else SC_TRY(tc ? tcgen05_branch_backward(ctx, b, S, n, sb[b]) : simt_branch_backward(ctx, b, S, n, sb[b]));
    if (b > 0) { SC_CUDA(cudaEventRecord(ev[3 + b], sb[b])); SC_CUDA(cudaStreamWaitEvent(st, ev[3 + b], 0)); }
  }
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// the step's persistent resources (allocated outside any stream capture)
static int step_prepare(sc_ctx* ctx, bool tc, bool head) {
  if (!ctx->train_consts) {
    SC_CUDA(cudaMalloc(&ctx->train_consts, 2 * kTrainZeros * sizeof(float)));
    std::vector<float> h1(2 * kTrainZeros);
    for (int i = 0; i < 2 * kTrainZeros; ++i) h1[i] = i < kTrainZeros ? 1.f : 0.f;
    SC_CUDA(cudaMemcpy(ctx->train_consts, h1.data(), h1.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  if (!ctx->train_side[0]) {
    for (int i = 0; i < 2; ++i) SC_CUDA(cudaStreamCreateWithFlags(&ctx->train_side[i], cudaStreamNonBlocking));
    for (int i = 0; i < 8; ++i) SC_CUDA(cudaEventCreateWithFlags(&ctx->train_ev[i], cudaEventDisableTiming));
  }
  if (tc && !head) SC_TRY(tc_train_prepare(ctx));
  if (tc) SC_TRY(tdense_prepare(ctx));
  return SC_OK;
}

// train_body on `st`, kernel by kernel or as the captured graph of its shape
static int run_step(sc_ctx* ctx, const StepBuf& S, int n, int64_t n_global, bool injected, cudaStream_t st) {
  const bool tc = ctx->gemm_backend == 1;
  const bool use_graph = ctx->train_graph_on && !ctx->profile && !(tc && ctx->ar_hook && !S.head);   // the sync-BN hook runs host code between kernels
  if (!use_graph) return train_body(ctx, S, n, n_global, injected, st);
  sc_ctx::TrainGraph key = {n, (long long)n_global, injected ? 1 : 0, ctx->gemm_backend, ctx->ws_fit.ptr, nullptr, 0,
                            {nullptr, nullptr, nullptr}, 0};
  if (S.head) {
    key.tables[0] = S.head->feats; key.tables[1] = S.head->atlas_rows; key.tables[2] = S.head->labels;
    key.has_idx = S.head->idx != nullptr;
  }
  sc_ctx::TrainGraph* g = nullptr;
  for (auto& e : ctx->train_graphs)
    if (e.n == key.n && e.n_global == key.n_global && e.injected == key.injected && e.backend == key.backend && e.arena == key.arena &&
        e.tables[0] == key.tables[0] && e.tables[1] == key.tables[1] && e.tables[2] == key.tables[2] && e.has_idx == key.has_idx) g = &e;
  if (!g) {
    // a moved arena invalidates every captured address
    for (size_t i = 0; i < ctx->train_graphs.size();) {
      if (ctx->train_graphs[i].arena != ctx->ws_fit.ptr) { cudaGraphExecDestroy(ctx->train_graphs[i].exec); ctx->train_graphs.erase(ctx->train_graphs.begin() + i); }
      else ++i;
    }
    if (ctx->train_graphs.size() >= 8) { cudaGraphExecDestroy(ctx->train_graphs[0].exec); ctx->train_graphs.erase(ctx->train_graphs.begin()); }
    cudaStream_t cap;
    SC_CUDA(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));   // capture on a private stream: `st` may be the legacy default stream
    const int64_t l0 = ctx->launches;
    SC_CUDA(cudaStreamBeginCapture(cap, cudaStreamCaptureModeRelaxed));
    const int bs = train_body(ctx, S, n, n_global, injected, cap);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(cap, &graph);
    cudaStreamDestroy(cap);
    const int launches = (int)(ctx->launches - l0);
    ctx->launches = l0;
    if (bs != SC_OK) { if (graph) cudaGraphDestroy(graph); return bs; }
    SC_CUDA(ce);
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    SC_CUDA(ie);
    key.exec = exec; key.launches = launches;
    ctx->train_graphs.push_back(key);
    g = &ctx->train_graphs.back();
  }
  SC_CUDA(cudaGraphLaunch(g->exec, st));
  ctx->launches += g->launches;
  return SC_OK;
}

int train_forward_backward(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, const float* in4, const uint8_t* y,
                           int64_t n64, int64_t n_global, uint64_t seed, const uint8_t* masks_in, float* loss, cudaStream_t st) {
  SC_CHECK(n64 <= 16384, SC_ERR_ARG, "sc_train_forward_backward: per-GPU batch %lld too large (max 16384)", (long long)n64);
  const int n = (int)n64;
  StepBuf S;
  const bool tc = ctx->gemm_backend == 1;
  const size_t need = carve_step(S, nullptr, n, tc);
  SC_TRY(ensure_ws(ctx->ws_fit, need + 4096));
  carve_step(S, reinterpret_cast<char*>(ctx->ws_fit.ptr), n, tc);
  SC_TRY(step_prepare(ctx, tc, false));
  // stage the caller's batch into the arena: the step itself only ever sees context-owned addresses
  const float* ins[3] = {in1, in2, in3};
  for (int b = 0; b < 3; ++b) SC_CUDA(cudaMemcpyAsync(S.in[b], ins[b], (size_t)n * 4096, cudaMemcpyDeviceToDevice, st));
  SC_CUDA(cudaMemcpyAsync(S.in4, in4, (size_t)n * 60, cudaMemcpyDeviceToDevice, st));
  SC_CUDA(cudaMemcpyAsync(S.y, y, (size_t)n, cudaMemcpyDeviceToDevice, st));
  if (masks_in) SC_CUDA(cudaMemcpyAsync(S.masks, masks_in, (size_t)n * 2700, cudaMemcpyDeviceToDevice, st));
  const unsigned long long seed_h = seed;
  SC_CUDA(cudaMemcpyAsync(S.seed, &seed_h, sizeof(seed_h), cudaMemcpyHostToDevice, st));   // pageable source: staged before the call returns
  // the split dense operands of the tcgen05 step: the step writes their valid entries only, the K padding must read as zero
  if (tc) SC_CUDA(cudaMemsetAsync(S.td.zero_begin, 0, S.td.zero_bytes, st));
  SC_TRY(run_step(ctx, S, n, n_global, masks_in != nullptr, st));
  SC_CUDA(cudaMemcpyAsync(loss, S.loss, sizeof(float), cudaMemcpyDeviceToDevice, st));
  return SC_OK;
}

// fine-tuning: one training step of the head (d1 x3, FC1, fc_2, out_layer) on rows idx[0..n) of a table of cached trunk
// features; the same dropout masks, loss and gradients as train_forward_backward with a trunk evaluated in deterministic mode
int head_train_forward_backward(sc_ctx* ctx, const float* feats, const float* atlas_rows, const uint8_t* labels, const int64_t* idx,
                                int64_t n64, int64_t n_global, uint64_t seed, const uint8_t* masks_in, float* loss, cudaStream_t st) {
  const int n = (int)n64;
  StepBuf S;
  const size_t need = carve_step(S, nullptr, n, true, true);
  SC_TRY(ensure_ws(ctx->ws_fit, need + 4096));
  carve_step(S, reinterpret_cast<char*>(ctx->ws_fit.ptr), n, true, true);
  SC_TRY(step_prepare(ctx, true, true));
  HeadGather g;
  g.feats = feats; g.atlas_rows = atlas_rows; g.labels = labels;
  g.idx = idx ? S.idx : nullptr; g.row0 = 0; g.n = n; g.masks = S.masks;
  for (int b = 0; b < 3; ++b) { g.F5s[b] = S.td.F5s[b]; g.F5T[b] = S.td.F5T[b]; }
  g.npad = S.td.npad; g.in4 = S.in4; g.y = S.y;
  S.head = &g;
  // per-step values: the index slice, the injected masks and the seed are staged into the arena (the tables are in the graph key)
  if (idx) SC_CUDA(cudaMemcpyAsync(S.idx, idx, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  if (masks_in) SC_CUDA(cudaMemcpyAsync(S.masks, masks_in, (size_t)n * 2700, cudaMemcpyDeviceToDevice, st));
  const unsigned long long seed_h = seed;
  SC_CUDA(cudaMemcpyAsync(S.seed, &seed_h, sizeof(seed_h), cudaMemcpyHostToDevice, st));   // pageable source: staged before the call returns
  SC_CUDA(cudaMemsetAsync(S.td.zero_begin, 0, S.td.zero_bytes, st));
  SC_TRY(run_step(ctx, S, n, n_global, masks_in != nullptr, st));
  SC_CUDA(cudaMemcpyAsync(loss, S.loss, sizeof(float), cudaMemcpyDeviceToDevice, st));
  return SC_OK;
}

// eval_fn: deterministic forward, sum of -log p[y] and number of correct arg-max
__global__ void eval_reduce_kernel(const float* __restrict__ proba, const uint8_t* __restrict__ y, int n, float* __restrict__ out2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.f, c = 0.f;
  if (i < n) {
    const float* p = proba + (int64_t)i * 15;
    int best = 0;
    for (int k = 1; k < 15; ++k) if (p[k] > p[best]) best = k;
    const int t = y[i] < 15 ? y[i] : 0;
    l = -logf(fmaxf(p[t], 1e-38f));
    c = best == t ? 1.f : 0.f;
  }
  for (int o = 16; o; o >>= 1) { l += __shfl_xor_sync(0xffffffffu, l, o); c += __shfl_xor_sync(0xffffffffu, c, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out2, l); atomicAdd(out2 + 1, c); }
}

int eval_batch(sc_ctx* ctx, const float* in1, const float* in2, const float* in3, const float* in4, const uint8_t* y, int64_t n,
               float* out2, cudaStream_t st) {
  SC_TRY(ensure_ws(ctx->ws_train, (size_t)n * 15 * sizeof(float) + 256));
  float* proba = reinterpret_cast<float*>(ctx->ws_train.ptr);
  SC_TRY(forward_patches(ctx, in1, in2, in3, in4, n, proba, nullptr, st));
  SC_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(float), st));
  return launch_eval_reduce(ctx, proba, y, n, out2, st);
}

int launch_eval_reduce(sc_ctx* ctx, const float* proba, const uint8_t* y, int64_t n, float* out2, cudaStream_t st) {
  eval_reduce_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(proba, y, (int)n, out2);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
