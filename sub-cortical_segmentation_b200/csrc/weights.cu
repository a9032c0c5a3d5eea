// Derived inference layouts from the pickle-ordered master parameters.
//
// Semantics being folded in (SURVEY.md 2.3; graph: cnn_cort/nets.py:170-231):
//   * Conv2DLayer flip_filters=True  -> taps are stored flipped so the kernels cross-correlate
//   * BatchNormLayer [beta,gamma,mean,inv_std] -> scale = gamma*inv_std, shift = beta - mean*scale
//   * DenseLayer W is (in, out); d1 flattens (c, h, w) -> k = c*9 + h*3 + w
//   * dense-dilated d1: a 3x3 dilation-4 conv over the NHWC-64 conv5 map, k = tap*64 + c (no flip)
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace sc {

static uint16_t bf16_rn(float x) {  // round to nearest even, like __float2bfloat16_rn
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static float bf16_to_float(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

struct Arena {
  std::vector<float> host;
  size_t alloc(size_t n) {
    size_t o = host.size();
    n = (n + 63) & ~(size_t)63;  // 256 B alignment for every array (TMA needs 16 B, float4 loads 16 B)
    host.resize(o + n, 0.f);
    return o;
  }
};

struct GemmOff { size_t kn, nk, bias, alpha, scale; };

static GemmOff make_gemm(Arena& A, GemmW& g, int K, int N, int Kpad, int Npad) {
  g.K = K; g.N = N; g.Kpad = Kpad; g.Npad = Npad;
  GemmOff o;
  o.kn = A.alloc((size_t)Kpad * Npad);
  o.nk = A.alloc((size_t)Npad * Kpad);
  o.bias = A.alloc(Npad);
  o.alpha = A.alloc(Npad);
  o.scale = A.alloc(Npad);
  for (int n = 0; n < Npad; ++n) { A.host[o.scale + n] = 1.f; A.host[o.alpha + n] = 1.f; }
  return o;
}
static void set_w(Arena& A, const GemmOff& o, const GemmW& g, int k, int n, float v) {
  A.host[o.kn + (size_t)k * g.Npad + n] = v;
  // split bf16 row: per 64-wide k block, 64 hi then 64 lo (2 bf16 per float slot of the arena)
  uint16_t* row = reinterpret_cast<uint16_t*>(&A.host[o.nk + (size_t)n * g.Kpad]);
  const uint16_t hi = bf16_rn(v);
  row[(k >> 6) * 128 + (k & 63)] = hi;
  row[(k >> 6) * 128 + 64 + (k & 63)] = bf16_rn(v - bf16_to_float(hi));
}
static void bind(GemmW& g, const GemmOff& o, float* base) {
  g.w_kn = base + o.kn; g.w_nk = base + o.nk; g.bias = base + o.bias; g.alpha = base + o.alpha; g.scale = base + o.scale;
}

int derive_weights(sc_ctx* ctx, cudaStream_t st) {
  const ParamOff& P = ctx->off;
  std::vector<float> h(P.total);
  SC_CUDA(cudaMemcpyAsync(h.data(), ctx->params, sizeof(float) * P.total, cudaMemcpyDeviceToHost, st));
  SC_CUDA(cudaStreamSynchronize(st));

  Arena A;
  struct BOff { size_t c1, conv[5], scale[5], shift[5], alpha[5], sw[5], swp[5]; GemmOff d1, d1d; } bo[3];
  GemmOff fc1o, fc2o;
  size_t outw, outb;
  for (int b = 0; b < 3; ++b) {
    const BranchOff& B = P.br[b];
    bo[b].c1 = A.alloc(9 * 20);
    for (int t = 0; t < 9; ++t)
      for (int co = 0; co < 20; ++co) A.host[bo[b].c1 + t * 20 + co] = ctx->br[b].c1_host.w[t * 20 + co] = h[B.convW[0] + co * 9 + (8 - t)];
    for (int l = 0; l < 5; ++l) {
      const int ci_n = kConvCin[l], co_n = kConvCout[l];
      if (l > 0) {
        bo[b].conv[l] = A.alloc((size_t)ci_n * 9 * co_n);
        for (int co = 0; co < co_n; ++co)
          for (int ci = 0; ci < ci_n; ++ci)
            for (int t = 0; t < 9; ++t)
              A.host[bo[b].conv[l] + ((size_t)ci * 9 + t) * co_n + co] = h[B.convW[l] + ((size_t)co * ci_n + ci) * 9 + (8 - t)];
      }
      bo[b].scale[l] = A.alloc(64);
      bo[b].shift[l] = A.alloc(64);
      bo[b].alpha[l] = A.alloc(64);
      if (l > 0) {   // strip-sweep kernel: k-step-packed weight panels, filter rows stacked, W hi rows then W lo rows
        SweepW& S = ctx->br[b].conv_sw[l];
        S.ksteps = (ci_n + 15) / 16; S.bn = (co_n + 15) & ~15; S.npanels = (3 * S.ksteps + 3) / 4;
        bo[b].sw[l] = A.alloc((size_t)S.npanels * 6 * S.bn * 32);
        bo[b].swp[l] = A.alloc((size_t)S.npanels * 6 * S.bn * 32);
        uint16_t* pw = reinterpret_cast<uint16_t*>(&A.host[bo[b].sw[l]]);
        uint16_t* pp = reinterpret_cast<uint16_t*>(&A.host[bo[b].swp[l]]);
        for (int co = 0; co < co_n; ++co)
          for (int ci = 0; ci < ci_n; ++ci)
            for (int t = 0; t < 9; ++t) {
              const float v = h[B.convW[l] + ((size_t)co * ci_n + ci) * 9 + (8 - t)];
              const uint16_t hi = bf16_rn(v), lo = bf16_rn(v - bf16_to_float(hi));
              size_t ip, iq;
              sweep_panel_pos(co, t / 3, t % 3, ci, S.ksteps, S.bn, ip, iq);
              pw[ip] = hi;
              pw[ip + (size_t)3 * S.bn * 64] = lo;
              pp[iq] = hi;
              pp[iq + (size_t)3 * S.bn / 2 * 64] = lo;
            }
      }
      for (int c = 0; c < co_n; ++c) {
        const float beta = h[B.bn[l][0] + c], gamma = h[B.bn[l][1] + c], mean = h[B.bn[l][2] + c], inv = h[B.bn[l][3] + c];
        const float s = gamma * inv;
        A.host[bo[b].scale[l] + c] = s;
        A.host[bo[b].shift[l] + c] = beta - mean * s;
        A.host[bo[b].alpha[l] + c] = h[B.alpha[l] + c];
        if (l == 0) { ctx->br[b].c1_host.scale[c] = s; ctx->br[b].c1_host.shift[c] = beta - mean * s; ctx->br[b].c1_host.alpha[c] = h[B.alpha[l] + c]; }
      }
    }
    bo[b].d1 = make_gemm(A, ctx->br[b].d1, 540, 180, kFeatLd, 192);
    bo[b].d1d = make_gemm(A, ctx->br[b].d1_dense, kD1K, 180, kD1K, 192);
    for (int k = 0; k < 540; ++k)
      for (int n = 0; n < 180; ++n) {
        const float v = h[B.d1W + (size_t)k * 180 + n];
        set_w(A, bo[b].d1, ctx->br[b].d1, k, n, v);
        const int c = k / 9, t = k % 9;
        set_w(A, bo[b].d1d, ctx->br[b].d1_dense, t * kC5Ld + c, n, v);
      }
    for (int n = 0; n < 192; ++n) {
      const float bias = n < 180 ? h[B.d1b + n] : 0.f, al = n < 180 ? h[B.d1alpha + n] : 1.f;
      A.host[bo[b].d1.bias + n] = A.host[bo[b].d1d.bias + n] = bias;
      A.host[bo[b].d1.alpha + n] = A.host[bo[b].d1d.alpha + n] = al;
    }
  }
  fc1o = make_gemm(A, ctx->fc1, 540, 540, kFeatLd, 576);
  for (int k = 0; k < 540; ++k)   // feature buffer: 192 columns per view (180 used) -> k' = view*192 + j
    for (int n = 0; n < 540; ++n) set_w(A, fc1o, ctx->fc1, (k / 180) * 192 + (k % 180), n, h[P.fc1W + (size_t)k * 540 + n]);
  for (int n = 0; n < 576; ++n) {
    A.host[fc1o.bias + n] = n < 540 ? h[P.fc1b + n] : 0.f;
    A.host[fc1o.alpha + n] = n < 540 ? h[P.a1 + n] : 1.f;
  }
  fc2o = make_gemm(A, ctx->fc2, 555, 270, kH1Ld, kH2Ld);
  ctx->fc2.k_used = 555;                     // h1 rows: 540 FC1 outputs | 15 atlas priors | zeros: the last k block needs 3 of its 4 k-steps
  for (int b = 0; b < 3; ++b) ctx->br[b].d1.k_used = 540;   // patchwise d1 over the flattened (c, h, w) features
  ctx->fc1.k_used = 0;                       // feature rows hold 192 columns per view (180 used): the last block is used up to column 563
  for (int k = 0; k < 555; ++k)
    for (int n = 0; n < 270; ++n) set_w(A, fc2o, ctx->fc2, k, n, h[P.fc2W + (size_t)k * 270 + n]);
  for (int n = 0; n < kH2Ld; ++n) {
    A.host[fc2o.bias + n] = n < 270 ? h[P.fc2b + n] : 0.f;
    A.host[fc2o.alpha + n] = n < 270 ? h[P.a2 + n] : 1.f;
  }
  outw = A.alloc(270 * 16);
  outb = A.alloc(16);
  for (int k = 0; k < 270; ++k)
    for (int n = 0; n < 15; ++n) A.host[outw + k * 16 + n] = h[P.outW + k * 15 + n];
  for (int n = 0; n < 15; ++n) A.host[outb + n] = h[P.outb + n];

  if (ctx->derived_floats < A.host.size()) {
    if (ctx->derived) cudaFree(ctx->derived);
    ctx->derived = nullptr;
    SC_CUDA(cudaMalloc(&ctx->derived, A.host.size() * sizeof(float)));
    ctx->derived_floats = A.host.size();
  }
  SC_CUDA(cudaMemcpyAsync(ctx->derived, A.host.data(), A.host.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  SC_CUDA(cudaStreamSynchronize(st));
  float* base = ctx->derived;
  for (int b = 0; b < 3; ++b) {
    ctx->br[b].c1_w = base + bo[b].c1;
    for (int l = 0; l < 5; ++l) {
      ctx->br[b].conv_w[l] = l > 0 ? base + bo[b].conv[l] : nullptr;
      ctx->br[b].scale[l] = base + bo[b].scale[l];
      ctx->br[b].shift[l] = base + bo[b].shift[l];
      ctx->br[b].alpha[l] = base + bo[b].alpha[l];
    }
    for (int l = 1; l < 5; ++l) {
      SweepW& S = ctx->br[b].conv_sw[l];
      S.panels = base + bo[b].sw[l]; S.panels_pair = base + bo[b].swp[l]; S.scale = ctx->br[b].scale[l]; S.shift = ctx->br[b].shift[l]; S.alpha = ctx->br[b].alpha[l];
    }
    bind(ctx->br[b].d1, bo[b].d1, base);
    bind(ctx->br[b].d1_dense, bo[b].d1d, base);
  }
  bind(ctx->fc1, fc1o, base);
  bind(ctx->fc2, fc2o, base);
  ctx->out_w = base + outw;
  ctx->out_b = base + outb;
  return SC_OK;
}

}  // namespace sc
