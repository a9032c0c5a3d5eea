// Dense layers of the training step on the tensor cores (d1 x3, FC1, fc_2, out_layer; cnn_cort/nets.py:179-231).
//
// Every contraction of the forward and backward pass is one launch of the split-bf16 tcgen05 GEMM of gemm_tc.cu
// (C[M][N] = A[M][K] * B[N][K]^T, both operands K-major rows of bf16 hi | lo blocks, fp32 accumulate):
//   forward   Z  [n][N]  = A  [n][K]  * W^T      B = W^T  [N][K]   (re-derived from the master parameters every step)
//   dgrad     dA [n][K]  = dZ [n][N]  * W        B = W    [K][N]   (the master layout itself, split)
//   wgrad     dW [K][N]  = A^T[K][n]  * dZ^T     B = dZ^T [N][n]   (the batch is the reduction axis)
// so each activation / gradient is kept twice: row-major split (next GEMM's A operand) and transposed split (the wgrad
// operands).  The element-wise kernels below (PReLU + dropout forward and backward, softmax cross-entropy, bias / slope
// gradients) write both copies.
#include "tc_common.cuh"

namespace sc {

__device__ __forceinline__ void put_split(float* base, int64_t row_floats, int64_t row, int col, float v) {
  __nv_bfloat16* r = reinterpret_cast<__nv_bfloat16*>(base + row * row_floats) + (col >> 6) * 128 + (col & 63);
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  r[0] = h;
  r[64] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// master W (K, N) row-major -> W^T [Npad][Kpad] split (forward B operand) and W [Krows][Npad64] split (dgrad B operand);
// bias -> zero-padded copy
__global__ void tderive_dense_kernel(const float* __restrict__ W, const float* __restrict__ bias, int K, int N, float* __restrict__ wnk, int Kpad,
                                     float* __restrict__ wkn, int Npad64, float* __restrict__ bias_pad, int Npad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Npad) bias_pad[i] = i < N ? bias[i] : 0.f;
  if (i >= K * N) return;
  const int k = i / N, n = i - k * N;
  const float v = W[i];
  put_split(wnk, Kpad, n, k, v);
  put_split(wkn, Npad64, k, n, v);
}

// v = act(in[m][j]) -> row-major split out[m][col0 + j] and transposed split outT[col0 + j][m].
// alpha != nullptr: PReLU; mask != nullptr: dropout keep-mask (x2).
__global__ void __launch_bounds__(256) tsplit_kernel(const float* __restrict__ in, int ld_in, int n, int N, const float* __restrict__ alpha,
                                                     const uint8_t* __restrict__ mask, int mask_ld, float* __restrict__ out, int ld_out, int col0,
                                                     float* __restrict__ outT, int npad) {
  const int64_t total = (int64_t)n * N;
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= total) return;
  auto value = [&](int m, int j) {
    float v = in[(int64_t)m * ld_in + j];
    if (alpha) v = prelu(v, alpha[j]);
    if (mask) v = mask[(int64_t)m * mask_ld + j] ? 2.f * v : 0.f;
    return v;
  };
  {  // j fastest: coalesced reads, row-major split writes
    const int m = (int)(e / N), j = (int)(e - (int64_t)m * N);
    put_split(out, ld_out, m, col0 + j, value(m, j));
  }
  {  // m fastest: contiguous transposed writes
    const int j = (int)(e / n), m = (int)(e - (int64_t)j * n);
    put_split(outT, npad, col0 + j, m, value(m, j));
  }
}

// softmax + cross-entropy on the [n][16] logits: dz = (p - onehot) / n_global as split rows [n][64] and transposed [16][npad];
// loss += sum(-log p[y]) / n_global
__global__ void tsoftmax_ce_kernel(const float* __restrict__ z, const uint8_t* __restrict__ y, int n, float inv_global, float* __restrict__ dz,
                                   float* __restrict__ dzT, int npad, float* __restrict__ gbias, float* __restrict__ loss) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.f;
  float d[15];
#pragma unroll
  for (int c = 0; c < 15; ++c) d[c] = 0.f;
  if (i < n) {
    float v[15], mx = -INFINITY, s = 0.f;
#pragma unroll
    for (int c = 0; c < 15; ++c) { v[c] = z[i * 16 + c]; mx = fmaxf(mx, v[c]); }
    const int t = y[i] < 15 ? y[i] : 0;
    const float zt = z[i * 16 + t] - mx;
#pragma unroll
    for (int c = 0; c < 15; ++c) { v[c] = expf(v[c] - mx); s += v[c]; }
    l = (logf(s) - zt) * inv_global;
#pragma unroll
    for (int c = 0; c < 15; ++c) {
      d[c] = (v[c] / s - (c == t ? 1.f : 0.f)) * inv_global;
      put_split(dz, 64, i, c, d[c]);
      put_split(dzT, npad, c, i, d[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < 15; ++c) {
    float sc_ = d[c];
    for (int o = 16; o; o >>= 1) sc_ += __shfl_xor_sync(0xffffffffu, sc_, o);
    if ((threadIdx.x & 31) == 0 && sc_ != 0.f) atomicAdd(&gbias[c], sc_);
  }
  for (int o = 16; o; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  if ((threadIdx.x & 31) == 0 && l != 0.f) atomicAdd(loss, l);
}

// PReLU (+ dropout) backward of a dense layer: dz = dy * (2 mask) * (z > 0 ? 1 : alpha) as split rows and transposed split;
// galpha[j] += sum_m dy' * z * [z <= 0]; gbias[j] += sum_m dz (the gradient buffer is cleared at the start of the step).
// One thread per element, visited twice like tsplit_kernel: j fastest for the row-major copy, m fastest for the transposed copy
// and the two column sums (a warp then holds 32 rows of one unit: shuffle reduction, one atomic per warp).
__global__ void __launch_bounds__(256) tsplit_bwd_kernel(const float* __restrict__ dy, int ld_dy, int col0, const float* __restrict__ z, int ldz, int n,
                                                         int N, const float* __restrict__ alpha, const uint8_t* __restrict__ mask, int mask_ld,
                                                         float* __restrict__ dz, int ld_dz, float* __restrict__ dzT, int npad,
                                                         float* __restrict__ galpha, float* __restrict__ gbias) {
  const int64_t total = (int64_t)n * N;
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const bool on = e < total;
  auto point = [&](int m, int j, float& g, float& zz) {
    g = dy[(int64_t)m * ld_dy + col0 + j];
    if (mask) g = mask[(int64_t)m * mask_ld + j] ? 2.f * g : 0.f;
    zz = z[(int64_t)m * ldz + j];
    return zz > 0.f ? g : alpha[j] * g;
  };
  if (on) {   // j fastest: coalesced reads, row-major split writes
    const int m = (int)(e / N), j = (int)(e - (int64_t)m * N);
    float g, zz;
    put_split(dz, ld_dz, m, j, point(m, j, g, zz));
  }
  int j2 = -1;
  float sa = 0.f, sb = 0.f;
  if (on) {   // m fastest: contiguous transposed writes, column sums
    j2 = (int)(e / n);
    const int m = (int)(e - (int64_t)j2 * n);
    float g, zz;
    const float d = point(m, j2, g, zz);
    put_split(dzT, npad, j2, m, d);
    if (zz <= 0.f) sa = g * zz;
    sb = d;
  }
  const int j0 = __shfl_sync(0xffffffffu, j2, 0);
  if (__all_sync(0xffffffffu, j2 == j0)) {
    for (int o = 16; o; o >>= 1) { sa += __shfl_xor_sync(0xffffffffu, sa, o); sb += __shfl_xor_sync(0xffffffffu, sb, o); }
    if ((threadIdx.x & 31) == 0 && j0 >= 0) { atomicAdd(&galpha[j0], sa); atomicAdd(&gbias[j0], sb); }
  } else if (on) {
    atomicAdd(&galpha[j2], sa); atomicAdd(&gbias[j2], sb);
  }
}

__global__ void tcopy_grad_kernel(const float* __restrict__ scratch, int ld, int K, int N, float* __restrict__ g) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K * N) return;
  const int k = i / N, j = i - k * N;
  g[i] = scratch[(int64_t)k * ld + j];
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static const int kDK[4] = {540, 540, 555, 270};      // fan-in of d1, FC1, fc_2, out_layer
static const int kDN[4] = {180, 540, 270, 15};       // fan-out
static const int kDKpad[4] = {576, 576, 576, 320};   // K padded to 64
static const int kDNpad[4] = {192, 576, 272, 16};    // rows of the forward B operand / columns of Z
static const int kDNpad64[4] = {192, 576, 320, 64};  // fan-out padded to 64 (K of the dgrad GEMM)

static size_t al1k(size_t v) { return (v + 1023) & ~(size_t)1023; }

size_t tdense_bytes(int n) {
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  size_t b = 0;
  // per branch: F5 split + T, Z1, dZ1 split + T, dF5, wgrad scratch
  b += 3 * (al1k((size_t)n * 576 * 4) + al1k(576 * npad * 4) + al1k((size_t)n * 192 * 4) + al1k((size_t)n * 192 * 4) + al1k(192 * npad * 4) +
            al1k((size_t)n * 576 * 4) + al1k((size_t)576 * 192 * 4));
  // head: CAT split + T, ZF1, CAT2 split + T, ZF2, H2 split + T, ZO, dZO split + T, dH2, dZF2 split + T, dCAT2, dZF1 split + T, dCAT
  b += 2 * (al1k((size_t)n * 576 * 4) + al1k(576 * npad * 4)) + al1k((size_t)n * 576 * 4) + al1k((size_t)n * 272 * 4) +
       al1k((size_t)n * 320 * 4) + al1k(320 * npad * 4) + al1k((size_t)n * 16 * 4) + al1k((size_t)n * 64 * 4) + al1k(16 * npad * 4) +
       al1k((size_t)n * 272 * 4) + al1k((size_t)n * 320 * 4) + al1k(272 * npad * 4) + al1k((size_t)n * 576 * 4) + al1k((size_t)n * 576 * 4) +
       al1k(576 * npad * 4) + al1k((size_t)n * 576 * 4);
  b += al1k((size_t)576 * 576 * 4) + al1k((size_t)576 * 272 * 4) + al1k((size_t)320 * 16 * 4);   // wgrad scratch of FC1, fc_2, out_layer
  return b + 64 * 1024;
}

void tdense_carve(TcDenseBuf& D, char* base, int n) {
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  size_t off = 0;
  auto take = [&](size_t bytes) { float* p = reinterpret_cast<float*>(base + off); off += al1k(bytes); return p; };
  D.npad = (int)npad;
  D.zero_begin = base;
  for (int b = 0; b < 3; ++b) {
    D.F5s[b] = take((size_t)n * 576 * 4); D.F5T[b] = take(576 * npad * 4);
    D.dZ1s[b] = take((size_t)n * 192 * 4); D.dZ1T[b] = take(192 * npad * 4);
  }
  D.CATs = take((size_t)n * 576 * 4); D.CATT = take(576 * npad * 4);
  D.CAT2s = take((size_t)n * 576 * 4); D.CAT2T = take(576 * npad * 4);
  D.H2s = take((size_t)n * 320 * 4); D.H2T = take(320 * npad * 4);
  D.dZOs = take((size_t)n * 64 * 4); D.dZOT = take(16 * npad * 4);
  D.dZF2s = take((size_t)n * 320 * 4); D.dZF2T = take(272 * npad * 4);
  D.dZF1s = take((size_t)n * 576 * 4); D.dZF1T = take(576 * npad * 4);
  D.zero_bytes = off;                                    // everything above has K padding that must read as zero
  for (int b = 0; b < 3; ++b) {
    D.Z1[b] = take((size_t)n * 192 * 4); D.dF5[b] = take((size_t)n * 576 * 4); D.gW1[b] = take((size_t)576 * 192 * 4);
  }
  D.ZF1 = take((size_t)n * 576 * 4); D.ZF2 = take((size_t)n * 272 * 4); D.ZO = take((size_t)n * 16 * 4);
  D.dH2 = take((size_t)n * 272 * 4); D.dCAT2 = take((size_t)n * 576 * 4); D.dCAT = take((size_t)n * 576 * 4);
  D.gWfc1 = take((size_t)576 * 576 * 4); D.gWfc2 = take((size_t)576 * 272 * 4); D.gWout = take((size_t)320 * 16 * 4);
}

// persistent device copies of the dense weights in the two operand layouts, re-derived every step
static int ensure_dense_weights(sc_ctx* ctx) {
  if (ctx->train_dense_w) return SC_OK;
  size_t total = 0;
  for (int t = 0; t < 6; ++t) {
    const int l = t < 3 ? 0 : t - 2;
    total += al1k((size_t)kDNpad[l] * kDKpad[l] * 4) + al1k((size_t)kDKpad[l] * kDNpad64[l] * 4) + al1k(1024 * 4);
  }
  SC_CUDA(cudaMalloc(&ctx->train_dense_w, total));
  SC_CUDA(cudaMemset(ctx->train_dense_w, 0, total));
  char* p = reinterpret_cast<char*>(ctx->train_dense_w);
  for (int t = 0; t < 6; ++t) {
    const int l = t < 3 ? 0 : t - 2;
    sc_ctx::TrainDenseW& W = ctx->train_dw[t];
    W.wnk = reinterpret_cast<float*>(p); p += al1k((size_t)kDNpad[l] * kDKpad[l] * 4);
    W.wkn = reinterpret_cast<float*>(p); p += al1k((size_t)kDKpad[l] * kDNpad64[l] * 4);
    W.bias = reinterpret_cast<float*>(p); p += al1k(1024 * 4);
  }
  return SC_OK;
}

int tdense_prepare(sc_ctx* ctx) { return ensure_dense_weights(ctx); }

static void master_of(const sc_ctx* ctx, int t, int& w, int& b) {
  const ParamOff& O = ctx->off;
  if (t < 3) { w = O.br[t].d1W; b = O.br[t].d1b; }
  else if (t == 3) { w = O.fc1W; b = O.fc1b; }
  else if (t == 4) { w = O.fc2W; b = O.fc2b; }
  else { w = O.outW; b = O.outb; }
}

int tdense_derive(sc_ctx* ctx, int t, cudaStream_t s) {
  SC_TRY(ensure_dense_weights(ctx));
  const int l = t < 3 ? 0 : t - 2;
  int w, b;
  master_of(ctx, t, w, b);
  const sc_ctx::TrainDenseW& W = ctx->train_dw[t];
  const int ne = kDK[l] * kDN[l];
  tderive_dense_kernel<<<(ne + 255) / 256, 256, 0, s>>>(ctx->params + w, ctx->params + b, kDK[l], kDN[l], W.wnk, kDKpad[l], W.wkn, kDNpad64[l],
                                                        W.bias, kDNpad[l]);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// C[M][ldc] (plain fp32) = A[M][K] * B[N][K]^T (+ bias); A, B split rows of K floats
static int tgemm(sc_ctx* ctx, const float* A, int M, int K, const float* B, int N, int Npad, const float* bias, float* C, int ldc, int n_store,
                 int cls, cudaStream_t s) {
  GemmW w;
  w.w_kn = nullptr; w.w_nk = const_cast<float*>(B); w.bias = const_cast<float*>(bias); w.alpha = ctx->train_consts;   // identity epilogue
  w.scale = nullptr; w.K = K; w.N = N; w.Kpad = K; w.Npad = Npad;
  GemmProblem p;
  gemm_problem_rows(p, A, K, K, M);
  p.C = C; p.ldc = ldc; p.n_store = n_store; p.out_split = 0; p.prof_cls = cls;
  return launch_gemm_tc(ctx, p, w, s);
}

static unsigned g256(int64_t total) { return (unsigned)((total + 255) / 256); }

int tdense_split(sc_ctx* ctx, const float* in, int ld_in, int n, int N, const float* alpha, const uint8_t* mask, float* out, int ld_out, int col0,
                 float* outT, int npad, cudaStream_t s) {
  tsplit_kernel<<<g256((int64_t)n * N), 256, 0, s>>>(in, ld_in, n, N, alpha, mask, 2700, out, ld_out, col0, outT, npad);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// d1 of branch b, forward: F5 (plain [n][540], dropout applied) -> CAT columns b*180.. (PReLU + f1_drop).  F5 == nullptr: the
// split operands D.F5s[b] / D.F5T[b] are already written (the head-only step gathers them from cached trunk features)
int tdense_branch_forward(sc_ctx* ctx, int b, const TcDenseBuf& D, const float* F5, int n, const uint8_t* masks, cudaStream_t s) {
  const BranchOff& Ob = ctx->off.br[b];
  SC_TRY(tdense_derive(ctx, b, s));
  if (F5) SC_TRY(tdense_split(ctx, F5, 540, n, 540, nullptr, nullptr, D.F5s[b], 576, 0, D.F5T[b], D.npad, s));
  SC_TRY(tgemm(ctx, D.F5s[b], n, 576, ctx->train_dw[b].wnk, 180, 192, ctx->train_dw[b].bias, D.Z1[b], 192, 180, PC_TRAIN_FWD, s));
  SC_TRY(tdense_split(ctx, D.Z1[b], 192, n, 180, ctx->params + Ob.d1alpha, masks + 1620 + b * 180, D.CATs, 576, b * 180, D.CATT, D.npad, s));
  return SC_OK;
}

// FC1 -> fc_2 -> out_layer -> softmax cross-entropy, then the backward pass of the head down to dCAT (plain [n][576])
int tdense_head(sc_ctx* ctx, const TcDenseBuf& D, const float* in4, const uint8_t* y, int n, int64_t n_global, const uint8_t* masks, float* loss,
                cudaStream_t s) {
  const ParamOff& O = ctx->off;
  float* P = ctx->params;
  float* G = ctx->grads;
  for (int t = 3; t < 6; ++t) SC_TRY(tdense_derive(ctx, t, s));
  const sc_ctx::TrainDenseW* W = ctx->train_dw;
  // ---- forward
  SC_TRY(tgemm(ctx, D.CATs, n, 576, W[3].wnk, 540, 576, W[3].bias, D.ZF1, 576, 540, PC_TRAIN_FWD, s));
  SC_TRY(tdense_split(ctx, D.ZF1, 576, n, 540, P + O.a1, masks + 2160, D.CAT2s, 576, 0, D.CAT2T, D.npad, s));
  SC_TRY(tdense_split(ctx, in4, 15, n, 15, nullptr, nullptr, D.CAT2s, 576, 540, D.CAT2T, D.npad, s));     // atlas priors: no dropout (nets.py:222-223)
  SC_TRY(tgemm(ctx, D.CAT2s, n, 576, W[4].wnk, 270, 272, W[4].bias, D.ZF2, 272, 272, PC_TRAIN_FWD, s));
  SC_TRY(tdense_split(ctx, D.ZF2, 272, n, 270, P + O.a2, nullptr, D.H2s, 320, 0, D.H2T, D.npad, s));
  SC_TRY(tgemm(ctx, D.H2s, n, 320, W[5].wnk, 15, 16, W[5].bias, D.ZO, 16, 16, PC_TRAIN_FWD, s));
  tsoftmax_ce_kernel<<<(n + 127) / 128, 128, 0, s>>>(D.ZO, y, n, 1.f / (float)n_global, D.dZOs, D.dZOT, D.npad, G + O.outb, loss);
  ctx->launches++;
  // ---- backward: out_layer
  SC_TRY(tgemm(ctx, D.H2T, 270, D.npad, D.dZOT, 15, 16, ctx->train_consts + kTrainZeros, D.gWout, 16, 16, PC_TRAIN_BWD, s));
  tcopy_grad_kernel<<<g256(270 * 15), 256, 0, s>>>(D.gWout, 16, 270, 15, G + O.outW);
  SC_TRY(tgemm(ctx, D.dZOs, n, 64, W[5].wkn, 270, 272, ctx->train_consts + kTrainZeros, D.dH2, 272, 272, PC_TRAIN_BWD, s));
  // fc_2
  tsplit_bwd_kernel<<<g256((int64_t)n * 270), 256, 0, s>>>(D.dH2, 272, 0, D.ZF2, 272, n, 270, P + O.a2, nullptr, 0, D.dZF2s, 320, D.dZF2T, D.npad,
                                                  G + O.a2, G + O.fc2b);
  SC_TRY(tgemm(ctx, D.CAT2T, 555, D.npad, D.dZF2T, 270, 272, ctx->train_consts + kTrainZeros, D.gWfc2, 272, 272, PC_TRAIN_BWD, s));
  tcopy_grad_kernel<<<g256(555 * 270), 256, 0, s>>>(D.gWfc2, 272, 555, 270, G + O.fc2W);
  SC_TRY(tgemm(ctx, D.dZF2s, n, 320, W[4].wkn, 555, 576, ctx->train_consts + kTrainZeros, D.dCAT2, 576, 556, PC_TRAIN_BWD, s));
  // FC1 (f2_drop sits on its activation)
  tsplit_bwd_kernel<<<g256((int64_t)n * 540), 256, 0, s>>>(D.dCAT2, 576, 0, D.ZF1, 576, n, 540, P + O.a1, masks + 2160, 2700, D.dZF1s, 576, D.dZF1T, D.npad,
                                                  G + O.a1, G + O.fc1b);
  SC_TRY(tgemm(ctx, D.CATT, 540, D.npad, D.dZF1T, 540, 576, ctx->train_consts + kTrainZeros, D.gWfc1, 576, 540, PC_TRAIN_BWD, s));
  tcopy_grad_kernel<<<g256(540 * 540), 256, 0, s>>>(D.gWfc1, 576, 540, 540, G + O.fc1W);
  SC_TRY(tgemm(ctx, D.dZF1s, n, 576, W[3].wkn, 540, 576, ctx->train_consts + kTrainZeros, D.dCAT, 576, 540, PC_TRAIN_BWD, s));
  ctx->launches += 5;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// d1 of branch b, backward: dCAT columns b*180.. -> gradients of d1 and (dgrad) dF5 (plain [n][576], columns 0..539)
int tdense_branch_backward(sc_ctx* ctx, int b, const TcDenseBuf& D, int n, const uint8_t* masks, bool dgrad, cudaStream_t s) {
  const BranchOff& Ob = ctx->off.br[b];
  float* P = ctx->params;
  float* G = ctx->grads;
  tsplit_bwd_kernel<<<g256((int64_t)n * 180), 256, 0, s>>>(D.dCAT, 576, b * 180, D.Z1[b], 192, n, 180, P + Ob.d1alpha, masks + 1620 + b * 180, 2700,
                                                  D.dZ1s[b], 192, D.dZ1T[b], D.npad, G + Ob.d1alpha, G + Ob.d1b);
  SC_TRY(tgemm(ctx, D.F5T[b], 540, D.npad, D.dZ1T[b], 180, 192, ctx->train_consts + kTrainZeros, D.gW1[b], 192, 180, PC_TRAIN_BWD, s));
  tcopy_grad_kernel<<<g256(540 * 180), 256, 0, s>>>(D.gW1[b], 192, 540, 180, G + Ob.d1W);
  if (dgrad)
    SC_TRY(tgemm(ctx, D.dZ1s[b], n, 192, ctx->train_dw[b].wkn, 540, 576, ctx->train_consts + kTrainZeros, D.dF5[b], 576, 540, PC_TRAIN_BWD, s));
  ctx->launches += 2;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
