// Whole-volume inference in the dense dilated formulation (SURVEY.md 8f-1).
//
// The reference evaluates the branch of cnn_cort/nets.py:170-180 on one 32x32 patch per
// candidate voxel (base.py:421-428).  Evaluated at EVERY pixel of a slice that is the same
// as running, on the slice zero-padded by (16 before, 15 after):
//   conv1 d=1 -> conv2 d=1 -> maxpool(2, stride 1) -> conv3 d=2 -> conv4 d=2 ->
//   maxpool(2, stride 1, dilation 2) -> conv5 d=4 -> d1 as a 3x3 dilation-4 conv (540 -> 180)
// (oracle/network.py:dense_branch proves the identity in fp64).  20x fewer FLOPs than the
// patchwise form and no patch materialisation at all.
//
// Coordinates: every layer buffer of a view shares the origin (r0, c0) of the requested
// output box in padded-slice coordinates; layer L covers rows [r0, r1 + ext_L):
//   ext: conv1 29, conv2 27, conv3 22, conv4 18, conv5 8, d1 0.
// This file: the orchestration (segment_volume, branch_patches_tc) and the fp32 SIMT back-end (planar maps
// [slice][C][rows][ld], pools folded into the load stage of conv3 / conv5, conv5 output NHWC-64 = the A operand of the d1
// implicit GEMM, K = tap*64 + c).  The default tensor-core back-end runs the conv layers in conv_sweep.cu (wide-row maps).
#include <thread>

#include "common.cuh"

namespace sc {


__host__ __device__ inline int round8(int v) { return (v + 7) & ~7; }

// ---------------------------------------------------------------------------------------
// conv1 (1 -> 20) straight from the volume, zero padding implicit.  4 pixels x 20 channels
// per thread; planar output.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dense_conv1_kernel(const float* __restrict__ vol, ViewGeo g, int sbeg, int ns,
                                                          const float* __restrict__ w, const float* __restrict__ scale,
                                                          const float* __restrict__ shift, const float* __restrict__ alpha,
                                                          float* __restrict__ out, int outR, int ld) {
  __shared__ float sw[9 * 20], ssc[20], ssh[20], sal[20];
  for (int i = threadIdx.x; i < 180; i += 256) sw[i] = w[i];
  if (threadIdx.x < 20) { ssc[threadIdx.x] = scale[threadIdx.x]; ssh[threadIdx.x] = shift[threadIdx.x]; sal[threadIdx.x] = alpha[threadIdx.x]; }
  __syncthreads();
  const int quads = ld >> 2;
  const int64_t total = (int64_t)ns * outR * quads;
  for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
    const int q = (int)(e % quads);
    const int i = (int)((e / quads) % outR);
    const int s = (int)(e / ((int64_t)quads * outR));
    const int j0 = q * 4;
    float x[3][6];
    const float* base = vol + (int64_t)(g.s0 + sbeg + s) * g.ss;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int rr = g.r0 + i + ky - 16;
      const bool rin = rr >= 0 && rr < g.R;
#pragma unroll
      for (int t = 0; t < 6; ++t) {
        const int cc = g.c0 + j0 + t - 16;
        x[ky][t] = (rin && cc >= 0 && cc < g.C) ? __ldg(base + (int64_t)rr * g.rs + (int64_t)cc * g.cs) : 0.f;
      }
    }
    float* o = out + (((int64_t)s * 20) * outR + i) * ld + j0;
    const int64_t plane = (int64_t)outR * ld;
#pragma unroll 4
    for (int co = 0; co < 20; ++co) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float wv = sw[(ky * 3 + kx) * 20 + co];
          a0 = fmaf(x[ky][kx + 0], wv, a0); a1 = fmaf(x[ky][kx + 1], wv, a1);
          a2 = fmaf(x[ky][kx + 2], wv, a2); a3 = fmaf(x[ky][kx + 3], wv, a3);
        }
      const float sc_ = ssc[co], sh = ssh[co], al = sal[co];
      float4 v;
      v.x = prelu(fmaf(a0, sc_, sh), al); v.y = prelu(fmaf(a1, sc_, sh), al);
      v.z = prelu(fmaf(a2, sc_, sh), al); v.w = prelu(fmaf(a3, sc_, sh), al);
      *reinterpret_cast<float4*>(o + co * plane) = v;
    }
  }
}

// ---------------------------------------------------------------------------------------
// conv2..conv5: 3x3 dilated conv + BN affine + PReLU over planar slices, fp32 FFMA.
// CTA = 320 threads = 64 pixel groups (16 rows x 4 segments of 8 columns) x 5 channel groups.
// Input channels stream through shared memory in chunks of 10 together with their taps.
// ---------------------------------------------------------------------------------------
template <int CIN, int COUT, int DIL, int POOLD, bool NHWC_OUT>
struct ConvCfg {
  static constexpr int TH = 16, TW = 32, CHUNK = 10;
  static constexpr int CO_T = COUT / 5;
  static constexpr int IH = TH + 2 * DIL;
  static constexpr int NV = (8 + 2 * DIL + 3) / 4;            // float4 loads per thread per input row
  static constexpr int IW = 24 + NV * 4;                      // widest column any thread reads
  static constexpr int IWP = (IW % 8 == 4) ? IW : IW + 4;     // row stride == 4 (mod 8): conflict-free LDS.128
  static constexpr int IN_FLOATS = CHUNK * IH * IWP;
  static constexpr int W_FLOATS = CHUNK * 9 * COUT;
  static constexpr size_t SMEM = (size_t)(IN_FLOATS + W_FLOATS) * sizeof(float);
};

template <int CIN, int COUT, int DIL, int POOLD, bool NHWC_OUT>
__global__ void __launch_bounds__(320) dense_conv_kernel(const ConvArgs a) {
  using Cfg = ConvCfg<CIN, COUT, DIL, POOLD, NHWC_OUT>;
  extern __shared__ __align__(16) float smem[];
  float* s_in = smem;
  float* s_w = smem + Cfg::IN_FLOATS;
  const int tid = threadIdx.x;
  const int cg = tid >> 6, pg = tid & 63, prow = pg >> 2, pseg = pg & 3;
  const int tr0 = blockIdx.y * Cfg::TH, tc0 = blockIdx.x * Cfg::TW;
  const int s = blockIdx.z;
  const float* in_s = a.in + (int64_t)s * CIN * a.inR * a.inLd;

  float acc[8][Cfg::CO_T];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int c = 0; c < Cfg::CO_T; ++c) acc[p][c] = 0.f;

  for (int ci0 = 0; ci0 < CIN; ci0 += Cfg::CHUNK) {
    __syncthreads();
    // stage CHUNK input planes (with the stride-1 max-pool of the previous layer folded in)
    for (int e = tid; e < Cfg::CHUNK * Cfg::IH * Cfg::IW; e += 320) {
      const int col = e % Cfg::IW;
      const int row = (e / Cfg::IW) % Cfg::IH;
      const int ci = e / (Cfg::IW * Cfg::IH);
      const int gr = tr0 + row, gc = tc0 + col;
      float v = 0.f;
      if (gr + POOLD < a.inR && gc + POOLD < a.inLd) {
        const float* p = in_s + ((int64_t)(ci0 + ci) * a.inR + gr) * a.inLd + gc;
        v = __ldg(p);
        if (POOLD > 0) {
          v = fmaxf(v, __ldg(p + POOLD));
          v = fmaxf(v, fmaxf(__ldg(p + (int64_t)POOLD * a.inLd), __ldg(p + (int64_t)POOLD * a.inLd + POOLD)));
        }
      }
      s_in[(ci * Cfg::IH + row) * Cfg::IWP + col] = v;
    }
    for (int e = tid; e < Cfg::W_FLOATS / 4; e += 320)
      reinterpret_cast<float4*>(s_w)[e] = __ldg(reinterpret_cast<const float4*>(a.w + (int64_t)ci0 * 9 * COUT) + e);
    __syncthreads();

#pragma unroll 1
    for (int ci = 0; ci < Cfg::CHUNK; ++ci) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        float x[Cfg::NV * 4];
        const float4* src = reinterpret_cast<const float4*>(s_in + (ci * Cfg::IH + prow + ky * DIL) * Cfg::IWP + pseg * 8);
#pragma unroll
        for (int v = 0; v < Cfg::NV; ++v) {
          const float4 t = src[v];
          x[v * 4 + 0] = t.x; x[v * 4 + 1] = t.y; x[v * 4 + 2] = t.z; x[v * 4 + 3] = t.w;
        }
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          float wv[Cfg::CO_T];
          const float4* wsrc = reinterpret_cast<const float4*>(s_w + (ci * 9 + ky * 3 + kx) * COUT + cg * Cfg::CO_T);
#pragma unroll
          for (int v = 0; v < Cfg::CO_T / 4; ++v) {
            const float4 t = wsrc[v];
            wv[v * 4 + 0] = t.x; wv[v * 4 + 1] = t.y; wv[v * 4 + 2] = t.z; wv[v * 4 + 3] = t.w;
          }
#pragma unroll
          for (int p = 0; p < 8; ++p)
#pragma unroll
            for (int c = 0; c < Cfg::CO_T; ++c) acc[p][c] = fmaf(x[kx * DIL + p], wv[c], acc[p][c]);
        }
      }
    }
  }

  const int orow = tr0 + prow, ocol = tc0 + pseg * 8;
  if (orow >= a.outR) return;
  if (!NHWC_OUT) {
    if (ocol >= a.outLd) return;
#pragma unroll
    for (int c = 0; c < Cfg::CO_T; ++c) {
      const int co = cg * Cfg::CO_T + c;
      const float sc_ = __ldg(a.scale + co), sh = __ldg(a.shift + co), al = __ldg(a.alpha + co);
      float r[8];
#pragma unroll
      for (int p = 0; p < 8; ++p) r[p] = prelu(fmaf(acc[p][c], sc_, sh), al);
      float* o = a.out + (((int64_t)s * COUT + co) * a.outR + orow) * a.outLd + ocol;
      *reinterpret_cast<float4*>(o) = make_float4(r[0], r[1], r[2], r[3]);
      *reinterpret_cast<float4*>(o + 4) = make_float4(r[4], r[5], r[6], r[7]);
    }
  } else {
    float sc_[Cfg::CO_T], sh[Cfg::CO_T], al[Cfg::CO_T];
#pragma unroll
    for (int c = 0; c < Cfg::CO_T; ++c) {
      const int co = cg * Cfg::CO_T + c;
      sc_[c] = __ldg(a.scale + co); sh[c] = __ldg(a.shift + co); al[c] = __ldg(a.alpha + co);
    }
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      if (ocol + p >= a.outC) break;
      float* o = a.out + (((int64_t)s * a.outR + orow) * a.outC + ocol + p) * kC5Ld;   // this pixel's 64-channel row
#pragma unroll
      for (int v = 0; v < Cfg::CO_T / 4; ++v) {
        float r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) r[k] = prelu(fmaf(acc[p][v * 4 + k], sc_[v * 4 + k], sh[v * 4 + k]), al[v * 4 + k]);
        store_row4(o, cg * Cfg::CO_T + v * 4, a.round_out, r[0], r[1], r[2], r[3]);
      }
      if (cg == 4 && COUT < kC5Ld) store_row4(o, COUT, a.round_out, 0.f, 0.f, 0.f, 0.f);
    }
  }
}

template <int CIN, int COUT, int DIL, int POOLD, bool NHWC_OUT>
static int launch_dense_conv(sc_ctx* ctx, const ConvArgs& a, int prof_cls, cudaStream_t st) {
  using Cfg = ConvCfg<CIN, COUT, DIL, POOLD, NHWC_OUT>;
  auto kern = dense_conv_kernel<CIN, COUT, DIL, POOLD, NHWC_OUT>;
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), (int)Cfg::SMEM));
  const int width = NHWC_OUT ? a.outC : a.outLd;
  dim3 grid((width + Cfg::TW - 1) / Cfg::TW, (a.outR + Cfg::TH - 1) / Cfg::TH, a.ns);
  ProfScope prof(ctx, prof_cls, st);
  kern<<<grid, 320, Cfg::SMEM, st>>>(a);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---------------------------------------------------------------------------------------
// Patchwise branch on the tensor cores (predict_proba on patch dicts)
// ---------------------------------------------------------------------------------------
// Patch maps in the wide-row layout of conv_sweep.cu: the patches of a chunk lie side by side, position
// (row r, patch p, col c) = r * (n * pitch) + p * pitch + c with pitch 32 / 16 / 8 per pooling level:
//   conv1 [30][n][32] F32CH -> conv2 + 2x2/2 pool [15][n][16] F32CH -> conv3 [15][n][16] F64CH
//   -> conv4 + 2x2/2 pool [7][n][8] F64CH -> conv5 [7][n][8] F64CH (3x3 valid) -> d1 reads its 9 taps through a 4-D tensor map
size_t branch_patches_tc_bytes(int64_t n) {
  return (size_t)n * ((960 + 240) * 32 + (240 + 56 + 56) * 64) * sizeof(float) + 5 * 256;
}

int branch_trunk_tc(sc_ctx* ctx, int b, const float* patches, int64_t n, float* scratch, float** c5_out, cudaStream_t st) {
  const BranchW& W = ctx->br[b];
  auto carve = [&](float*& cur, size_t floats) { float* p = cur; cur += (floats + 63) & ~(size_t)63; return p; };
  float* cur = scratch;
  float* c1 = carve(cur, (size_t)n * 960 * 32);
  float* p1 = carve(cur, (size_t)n * 240 * 32);
  float* c3 = carve(cur, (size_t)n * 240 * 64);
  float* p2 = carve(cur, (size_t)n * 56 * 64);
  float* c5 = carve(cur, (size_t)n * 56 * 64);
  SC_CHECK(n * 960 < (1ll << 31), SC_ERR_ARG, "patchwise chunk too large");
  {
    ViewGeo g = {1024, 32, 1, 0, (int)n, 16, 16, 30, 30, 32, 32};   // origin 16 cancels the dense path's zero-pad offset
    SC_TRY(launch_conv1_wide(ctx, patches, g, (int)n, W.c1_host, c1, 30, 32, st));
  }
  SC_TRY(launch_conv_sweep(ctx, W.conv_sw[1], 1, c1, 1, p1, 1, (int)(n * 32), 30, 28, 1, 2, PC_CONV2, st));   // conv2 + pool1 -> [15][n][16]
  SC_TRY(launch_conv_sweep(ctx, W.conv_sw[2], 2, p1, 1, c3, 0, (int)(n * 16), 15, 12, 1, 0, PC_CONV3, st));   // conv3
  SC_TRY(launch_conv_sweep(ctx, W.conv_sw[3], 3, c3, 0, p2, 0, (int)(n * 16), 15, 10, 1, 2, PC_CONV4, st));   // conv4 + pool2 -> [7][n][8]
  SC_TRY(launch_conv_sweep(ctx, W.conv_sw[4], 4, p2, 0, c5, 0, (int)(n * 8), 7, 3, 1, 0, PC_CONV5, st));     // conv5
  *c5_out = c5;
  return SC_OK;
}

int branch_patches_tc(sc_ctx* ctx, int b, const float* patches, int64_t n, float* scratch, float* feats, cudaStream_t st) {
  float* c5 = nullptr;
  SC_TRY(branch_trunk_tc(ctx, b, patches, n, scratch, &c5, st));
  // d1: rows = patches; tap (ty, tx) of the 3x3 conv5 map is tensor-map coordinate (k, patch, tx, ty); K = tap*64 + c
  GemmProblem p;
  p.A = c5; p.lda = 8 * kC5Ld; p.a_ys = 0; p.a_zs = 0;
  p.ntaps = 9; p.kc = kC5Ld; p.k_used = 0;
  for (int t = 0; t < 9; ++t) {
    p.tap_dx[t] = 0; p.tap_dy[t] = t % 3; p.tap_dz[t] = t / 3;
    p.tap_off[t] = ((int64_t)(t / 3) * n * 8 + (t % 3)) * kC5Ld;
  }
  p.a_base = c5; p.a_dims[0] = kC5Ld; p.a_dims[1] = n; p.a_dims[2] = 8; p.a_dims[3] = 7;
  p.a_strides[0] = 8 * kC5Ld; p.a_strides[1] = kC5Ld; p.a_strides[2] = (int64_t)n * 8 * kC5Ld;
  p.a_y0 = p.a_z0 = 0;
  p.C = feats; p.ldc = kFeatLd; p.c_ys = p.c_zs = 0; p.M = (int)n; p.Y = p.Z = 1;
  p.n_store = 192; p.c_col0 = b * 192; p.out_split = 1; p.prof_cls = PC_GEMM_D1;
  SC_TRY(launch_gemm_tc(ctx, p, ctx->br[b].d1_dense, st));
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// plain (dilation 1, no folded pool, planar) 3x3 valid conv over [n][CIN][R][ld] maps: the training
// forward convs and -- with the roles of the channel axes swapped and raw taps -- their dgrads.
int launch_conv3x3(sc_ctx* ctx, int cin, int cout, const ConvArgs& a, int prof_cls, cudaStream_t st) {
  if (cin == 20 && cout == 20) return launch_dense_conv<20, 20, 1, 0, false>(ctx, a, prof_cls, st);
  if (cin == 20 && cout == 40) return launch_dense_conv<20, 40, 1, 0, false>(ctx, a, prof_cls, st);
  if (cin == 40 && cout == 40) return launch_dense_conv<40, 40, 1, 0, false>(ctx, a, prof_cls, st);
  if (cin == 40 && cout == 60) return launch_dense_conv<40, 60, 1, 0, false>(ctx, a, prof_cls, st);
  if (cin == 60 && cout == 40) return launch_dense_conv<60, 40, 1, 0, false>(ctx, a, prof_cls, st);
  if (cin == 40 && cout == 20) return launch_dense_conv<40, 20, 1, 0, false>(ctx, a, prof_cls, st);
  set_error("launch_conv3x3: unsupported channel pair %d -> %d", cin, cout);
  return SC_ERR_ARG;
}

// conv1 (1 -> 20) over [n][32][32] patches -> planar [n][20][30][32]
int launch_conv1_patches(sc_ctx* ctx, const float* patches, int n, const float* w, const float* scale, const float* shift,
                         const float* alpha, float* out, cudaStream_t st) {
  ViewGeo g = {1024, 32, 1, 0, n, 16, 16, 30, 30, 32, 32};  // origin 16 cancels the dense path's zero-pad offset
  const int64_t work = (int64_t)n * 30 * 8;
  const int64_t blocks = (work + 255) / 256;
  const unsigned grid = (unsigned)(blocks < (int64_t)ctx->sm_count * 32 ? blocks : (int64_t)ctx->sm_count * 32);
  ProfScope prof(ctx, PC_TRAIN_FWD, st);
  dense_conv1_kernel<<<grid, 256, 0, st>>>(patches, g, 0, n, w, scale, shift, alpha, out, 30, 32);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// atlas prior (with the background fix of base.py:392-394) -> columns 540..575 of the h1 rows
__global__ void dense_atlas_kernel(const float* __restrict__ atlas, OutGeo g, int ix0, int64_t rows, float* __restrict__ h1,
                                   int split) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= rows) return;
  const int64_t plane = (int64_t)g.by * g.bz;
  const int ix = (int)(m / plane);
  const int rem = (int)(m - (int64_t)ix * plane);
  const int iy = rem / g.bz, iz = rem - iy * g.bz;
  const int64_t v = ((int64_t)(g.x0 + ix0 + ix) * g.Y + (g.y0 + iy)) * g.Z + (g.z0 + iz);
  float a[16];
#pragma unroll
  for (int c = 0; c < 15; ++c) a[c] = __ldg(atlas + v * 15 + c);
  float s = __fadd_rn(__fadd_rn(__fadd_rn(a[0], a[1]), __fadd_rn(a[2], a[3])),
                      __fadd_rn(__fadd_rn(a[4], a[5]), __fadd_rn(a[6], a[7])));
#pragma unroll
  for (int k = 8; k < 15; ++k) s = __fadd_rn(s, a[k]);
  if (s == 0.f) a[14] = 1.f;
  a[15] = 0.f;
  float* hr = h1 + m * kH1Ld;
#pragma unroll
  for (int q = 0; q < 9; ++q) {
    if (q < 4) store_row4(hr, 540 + 4 * q, split, a[4 * q], a[4 * q + 1], a[4 * q + 2], a[4 * q + 3]);
    else store_row4(hr, 540 + 4 * q, split, 0.f, 0.f, 0.f, 0.f);
  }
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

int segment_volume(sc_ctx* ctx, const float* vol, const int32_t* dims, const float* atlas, const int32_t* box,
                   const uint8_t* cand, uint8_t* label_vol, float* proba_vol, cudaStream_t st, const McArgs* mc) {
  const int X = dims[0], Y = dims[1], Z = dims[2];
  int b[6] = {0, X, 0, Y, 0, Z};
  if (box) for (int i = 0; i < 6; ++i) b[i] = box[i];
  SC_CHECK(b[0] >= 0 && b[1] <= X && b[2] >= 0 && b[3] <= Y && b[4] >= 0 && b[5] <= Z, SC_ERR_ARG, "sc_segment_volume: box outside the volume");
  const int bx = b[1] - b[0], by = b[3] - b[2], bz = b[5] - b[4];
  if (bx <= 0 || by <= 0 || bz <= 0) return SC_OK;
  const int64_t YZ = (int64_t)Y * Z;
  const bool tc = ctx->gemm_backend == 1;
  SC_CHECK(!mc || tc, SC_ERR_ARG, "segment_volume: Monte-Carlo dropout needs the tcgen05 back-end");

  ViewGeo vg[3];
  // axial: slices along z, rows x, cols y  (patch axes (dx, dy), base.py:291-292)
  vg[0] = {1, YZ, Z, b[4], bz, b[0], b[2], bx, by, X, Y};
  // coronal: slices along y, rows x, cols z
  vg[1] = {Z, YZ, 1, b[2], by, b[0], b[4], bx, bz, X, Z};
  // saggital: slices along x, rows y, cols z
  vg[2] = {YZ, Z, 1, b[0], bx, b[2], b[4], by, bz, Y, Z};

  // ---- workspace carve-up ----------------------------------------------------------------
  size_t a5_off[3], a5_bytes = 0;
  for (int v = 0; v < 3; ++v) {
    a5_off[v] = a5_bytes;
    // tensor-core mode: every map of a view is a flattened pixel sequence with the conv1 geometry (rows br+29, pitch bc+29)
    a5_bytes += tc ? align256((size_t)vg[v].ns * (vg[v].br + 29) * (vg[v].bc + 29) * kC5Ld * sizeof(float))
                   : align256((size_t)vg[v].ns * (vg[v].br + 8) * (vg[v].bc + 8) * kC5Ld * sizeof(float));
  }
  size_t per_slice_max = 0, view_max = 0;
  for (int v = 0; v < 3; ++v) {
    const size_t br = vg[v].br, bc = vg[v].bc;
    size_t f;
    if (tc) {  // strip-sweep pipeline: whole-view wide-row maps conv1 and pool1 (128 B pixels), conv3, pool2 (256 B pixels)
      f = (size_t)vg[v].ns * (br + 29) * (bc + 29) * (2 * 32 + 2 * 64) + 4 * 64;
      view_max = f > view_max ? f : view_max;
      continue;
    }
    f = 20 * (br + 29) * round8(bc + 29) + 20 * (br + 27) * round8(bc + 27) + 40 * (br + 22) * round8(bc + 22) +
        40 * (br + 18) * round8(bc + 18);
    per_slice_max = f > per_slice_max ? f : per_slice_max;
  }
  const size_t scratch_budget = (size_t)1536 << 20;
  int group = tc ? 1 : (int)(scratch_budget / (per_slice_max * sizeof(float) + 1024));
  if (group < 1) group = 1;
  if (group > 64) group = 64;
  const size_t scratch_bytes = tc ? align256(view_max * sizeof(float) + 4096) : align256((per_slice_max * sizeof(float) + 1024) * group);
  const int64_t plane = (int64_t)by * bz;
  int slab = (int)(ctx->chunk_voxels / plane);
  if (slab < 1) slab = 1;
  if (slab > bx) slab = bx;
  const size_t rows_max = (size_t)slab * plane;
  const size_t feat_bytes = align256(rows_max * kFeatLd * sizeof(float));
  const size_t h1_bytes = align256(rows_max * kH1Ld * sizeof(float));
  const size_t h2_bytes = tc ? 0 : align256(rows_max * kH2Ld * sizeof(float));   // tensor-core mode: fc_2 feeds the out_layer in its epilogue
  // candidate compaction (tensor-core path with a mask): the FC head runs on the candidate rows of each slab only
  const int nslabs = (bx + slab - 1) / slab;
  bool compact = tc && cand != nullptr && ctx->tc_compact && nslabs <= 4096;
  const size_t nbox = (size_t)bx * plane;
  const size_t cmp_blocks = (size_t)nslabs * ((rows_max + 2047) / 2048);
  const size_t cmp_bytes = compact ? align256(nbox * 4) * 2 + align256(cmp_blocks * 8 + 16) + align256((size_t)nslabs * 4) : 0;
  // sparse masks: per-view candidate occupancy (one 32-bit word per (row, slice)) + the item flags of one sweep launch
  size_t occ_off[3], skip_bytes = 0;
  for (int v = 0; v < 3; ++v) { occ_off[v] = skip_bytes; skip_bytes += compact ? align256((size_t)vg[v].br * vg[v].ns * 4) : 0; }
  const size_t flags_off = skip_bytes;
  if (compact) skip_bytes += align256((size_t)1 << 20);
  const size_t mc_bytes = mc ? align256(rows_max * 16 * sizeof(float)) : 0;   // Monte-Carlo dropout: 16 sums per FC row
  const size_t total = a5_bytes + scratch_bytes + feat_bytes + h1_bytes + h2_bytes + cmp_bytes + mc_bytes + skip_bytes;
  SC_TRY(ensure_ws(ctx->ws, total));
  char* wsb = reinterpret_cast<char*>(ctx->ws.ptr);
  float* a5[3] = {reinterpret_cast<float*>(wsb + a5_off[0]), reinterpret_cast<float*>(wsb + a5_off[1]),
                  reinterpret_cast<float*>(wsb + a5_off[2])};
  char* scratch = wsb + a5_bytes;
  float* feats = reinterpret_cast<float*>(scratch + scratch_bytes);
  float* h1 = reinterpret_cast<float*>(reinterpret_cast<char*>(feats) + feat_bytes);
  float* h2 = reinterpret_cast<float*>(reinterpret_cast<char*>(h1) + h1_bytes);
  int32_t* rowmap = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(h2) + h2_bytes);
  int32_t* rowvox = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(rowmap) + align256(nbox * 4));
  int32_t* cmp_scratch = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(rowvox) + align256(nbox * 4));
  int32_t* d_slab_cnt = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(cmp_scratch) + align256(cmp_blocks * 8 + 16));
  float* mc_acc = reinterpret_cast<float*>(wsb + (total - skip_bytes - mc_bytes));
  char* skip_base = wsb + (total - skip_bytes);
  if (compact) {
    // enqueue the scan first: its (tiny) result is on the host long before phase 1 has been launched
    if (!ctx->h_slab_cnt) {
      SC_CUDA(cudaMallocHost(&ctx->h_slab_cnt, 4096 * sizeof(int32_t)));
      SC_CUDA(cudaEventCreateWithFlags(&ctx->compact_ev, cudaEventDisableTiming));
    }
    OutGeo boxg = {b[0], b[2], b[4], by, bz, Y, Z};
    SC_TRY(launch_slab_compact(ctx, cand, boxg, bx, slab, rowmap, rowvox, d_slab_cnt, cmp_scratch, st));
    SC_CUDA(cudaMemcpyAsync(ctx->h_slab_cnt, d_slab_cnt, (size_t)nslabs * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    SC_CUDA(cudaEventRecord(ctx->compact_ev, st));
    // the candidate count decides both the compaction of the FC head and whether the sweeps skip items: one short wait here
    SC_CUDA(cudaEventSynchronize(ctx->compact_ev));
    int64_t ncand = 0;
    for (int i = 0; i < nslabs; ++i) ncand += ctx->h_slab_cnt[i];
    if (ncand * 10 >= (int64_t)nbox * 9) compact = false;     // (nearly) every voxel is a candidate: the dense rows are cheaper
  }
  // sparse mask: the sweeps only compute the items (strip x row segment) within the receptive-field reach of a candidate
  SweepSkip skips[3];
  const bool skip_on = compact && ctx->tc_skip;
  if (skip_on) {
    for (int v = 0; v < 3; ++v) {
      uint32_t* occ = reinterpret_cast<uint32_t*>(skip_base + occ_off[v]);
      SC_TRY(launch_view_occupancy(ctx, cand, vg[v], occ, st));
      skips[v] = {occ, vg[v].br, vg[v].bc, vg[v].ns, vg[v].bc + 29, reinterpret_cast<uint8_t*>(skip_base + flags_off)};
    }
  }

  // ---- phase 1: conv1..conv5 per view, slices in groups ------------------------------------
  for (int v = 0; v < 3; ++v) {
    const ViewGeo& g = vg[v];
    const BranchW& W = ctx->br[v];
    const int r1 = g.br + 29, l1 = round8(g.bc + 29);
    const int r2 = g.br + 27, l2 = round8(g.bc + 27);
    const int r3 = g.br + 22, l3 = round8(g.bc + 22);
    const int r4 = g.br + 18, l4 = round8(g.bc + 18);
    const int r5 = g.br + 8, c5 = g.bc + 8;
    if (tc) {
      // ---- tensor-core pipeline (conv_sweep.cu): whole-view wide-row maps, position = (row * ns + slice) * C1 + col, all
      // with the conv1 geometry (R1 rows, C1 columns per slice).  Positions outside a layer's valid region hold garbage
      // that valid outputs never read.  Every layer is a strip sweep (every input row loaded once, pools fused into the
      // epilogues); conv4 + pool2 and conv5 run on CTA pairs.
      const int R1 = g.br + 29, C1 = g.bc + 29;
      const int64_t Pw64 = (int64_t)g.ns * C1;
      const int64_t npos = Pw64 * R1;
      SC_CHECK(npos < (1ll << 31), SC_ERR_ARG, "sc_segment_volume: view too large");
      const int Pw = (int)Pw64;
      auto carve = [&](float*& cur, int px_floats) { float* p = cur; cur += align256((size_t)npos * px_floats * 4) / 4; return p; };
      float* cur = reinterpret_cast<float*>(scratch);
      float* m1 = carve(cur, 32); float* mp1 = carve(cur, 32);
      float* m3 = carve(cur, 64); float* mp2 = carve(cur, 64);
      SC_TRY(launch_conv1_wide(ctx, vol, g, g.ns, W.c1_host, m1, R1, C1, st));
      const SweepSkip* sk = skip_on ? &skips[v] : nullptr;
      SC_TRY(launch_conv_sweep(ctx, W.conv_sw[1], 1, m1, 1, mp1, 1, Pw, R1, g.br + 26, 1, 1, PC_CONV2, st, 0, 0, sk));     // conv2 + pool1
      SC_TRY(launch_conv_sweep(ctx, W.conv_sw[2], 2, mp1, 1, m3, 0, Pw, R1, g.br + 22, 2, 0, PC_CONV3, st, 0, 0, sk));     // conv3
      SC_TRY(launch_conv_sweep(ctx, W.conv_sw[3], 3, m3, 0, mp2, 0, Pw, R1, g.br + 16, 2, 1, PC_CONV4, st, 0, 0, sk));     // conv4 + pool2 (CTA pairs)
      SC_TRY(launch_conv_sweep(ctx, W.conv_sw[4], 4, mp2, 0, a5[v], 0, Pw, R1, g.br + 8, 4, 0, PC_CONV5, st, 0, 0, sk));   // conv5 (CTA pairs)
      SC_CUDA(cudaGetLastError());
    }
    for (int sb = 0; sb < g.ns && !tc; sb += group) {
      const int ns = g.ns - sb < group ? g.ns - sb : group;
      float* c1 = reinterpret_cast<float*>(scratch);
      float* c2 = c1 + align256((size_t)ns * 20 * r1 * l1 * 4) / 4;
      float* c3 = c2 + align256((size_t)ns * 20 * r2 * l2 * 4) / 4;
      float* c4 = c3 + align256((size_t)ns * 40 * r3 * l3 * 4) / 4;
      {
        const int64_t work = (int64_t)ns * r1 * (l1 / 4);
        const int64_t blocks = (work + 255) / 256;
        const unsigned grid = (unsigned)(blocks < (int64_t)ctx->sm_count * 32 ? blocks : (int64_t)ctx->sm_count * 32);
        ProfScope prof(ctx, PC_CONV1, st);
        dense_conv1_kernel<<<grid, 256, 0, st>>>(vol, g, sb, ns, W.c1_w, W.scale[0], W.shift[0], W.alpha[0], c1, r1, l1);
        ctx->launches++;
        SC_CUDA(cudaGetLastError());
      }
      ConvArgs a;
      a.ns = ns; a.round_out = 0;
      a.in = c1; a.inR = r1; a.inLd = l1; a.out = c2; a.outR = r2; a.outC = g.bc + 27; a.outLd = l2;
      a.w = W.conv_w[1]; a.scale = W.scale[1]; a.shift = W.shift[1]; a.alpha = W.alpha[1];
      SC_TRY((launch_dense_conv<20, 20, 1, 0, false>(ctx, a, PC_CONV2, st)));
      a.in = c2; a.inR = r2; a.inLd = l2; a.out = c3; a.outR = r3; a.outC = g.bc + 22; a.outLd = l3;
      a.w = W.conv_w[2]; a.scale = W.scale[2]; a.shift = W.shift[2]; a.alpha = W.alpha[2];
      SC_TRY((launch_dense_conv<20, 40, 2, 1, false>(ctx, a, PC_CONV3, st)));
      a.in = c3; a.inR = r3; a.inLd = l3; a.out = c4; a.outR = r4; a.outC = g.bc + 18; a.outLd = l4;
      a.w = W.conv_w[3]; a.scale = W.scale[3]; a.shift = W.shift[3]; a.alpha = W.alpha[3];
      SC_TRY((launch_dense_conv<40, 40, 2, 0, false>(ctx, a, PC_CONV4, st)));
      a.in = c4; a.inR = r4; a.inLd = l4; a.out = a5[v] + (size_t)sb * r5 * c5 * kC5Ld; a.outR = r5; a.outC = c5; a.outLd = c5;
      a.w = W.conv_w[4]; a.scale = W.scale[4]; a.shift = W.shift[4]; a.alpha = W.alpha[4];
      a.round_out = tc ? 1 : 0;
      SC_TRY((launch_dense_conv<40, 60, 4, 2, true>(ctx, a, PC_CONV5, st)));
    }
  }

  // ---- phase 2: d1 (x3) + FC head per slab of x-planes -------------------------------------
  int atlas_waited = 0;                                // chunked upload: chunks of x-planes this stream has already waited for
  const int passes = mc ? mc->samples : 1;
  McWeights mcw;
  if (mc) SC_TRY(mc_prepare(ctx, mcw));
  OutGeo og = {b[0], b[2], b[4], by, bz, Y, Z};
  for (int ix0 = 0; ix0 < bx; ix0 += slab) {
    const int nx = bx - ix0 < slab ? bx - ix0 : slab;
    const int64_t rows = (int64_t)nx * plane;
    if (ctx->atlas_chunks > 0) {                       // the atlas planes of this slab must have arrived
      int need = (b[0] + ix0 + nx + ctx->atlas_chunk_nx - 1) / ctx->atlas_chunk_nx;
      if (need > ctx->atlas_chunks) need = ctx->atlas_chunks;
      if (need > atlas_waited) {
        if (ctx->atlas_recorded)       // pageable upload by a helper thread: the event must have been recorded first
          while (ctx->atlas_recorded->load(std::memory_order_acquire) < need) std::this_thread::yield();
        SC_CUDA(cudaStreamWaitEvent(st, ctx->atlas_chunk_ev[need - 1], 0));
        atlas_waited = need;
      }
    }
    const int64_t slab_base = (int64_t)ix0 * plane;
    const int64_t rows_fc = compact ? ctx->h_slab_cnt[ix0 / slab] : rows;      // rows of the FC head (compact: candidates only)
    if (rows_fc == 0) continue;
    // Monte-Carlo dropout: the FC head once per pass with the row-masked weights of that pass (mc_dropout.cu)
    for (int pass = 0; pass < passes; ++pass) {
      if (mc) SC_TRY(launch_mc_mask(ctx, mc->seed, pass, st));
      for (int v = 0; v < 3; ++v) {
        const ViewGeo& g = vg[v];
        const int64_t c5 = tc ? g.bc + 29 : g.bc + 8, r5 = tc ? g.br + 29 : g.br + 8;   // tensor-core mode: conv1 geometry (see phase 1)
        GemmProblem p;
        p.lda = kC5Ld; p.a_ys = c5 * kC5Ld; p.a_zs = r5 * c5 * kC5Ld;
        p.ntaps = 9; p.kc = kC5Ld;
        for (int t = 0; t < 9; ++t) {
          p.tap_off[t] = ((int64_t)(t / 3) * 4 * c5 + (t % 3) * 4) * kC5Ld;
          p.tap_dx[t] = (t % 3) * 4; p.tap_dy[t] = (t / 3) * 4;
        }
        p.a_base = a5[v]; p.a_dims[0] = kC5Ld; p.a_dims[1] = c5; p.a_dims[2] = r5; p.a_dims[3] = g.ns;
        p.a_strides[0] = kC5Ld; p.a_strides[1] = c5 * kC5Ld; p.a_strides[2] = r5 * c5 * kC5Ld;
        p.a_swap = 0;
        if (tc) {   // wide-row map: (k, col, slice, row) with strides (pixel, C1 pixels, ns * C1 pixels)
          p.a_dims[2] = g.ns; p.a_dims[3] = r5;
          p.a_strides[1] = c5 * kC5Ld; p.a_strides[2] = (int64_t)g.ns * c5 * kC5Ld;
          p.a_swap = 1;
        }
        p.a_y0 = v == 2 ? 0 : ix0; p.a_z0 = v == 2 ? ix0 : 0;
        p.ldc = 0; p.out_split = tc ? 1 : 0; p.c_col0 = v * 192; p.prof_cls = PC_GEMM_D1; p.k_used = 0;
        p.n_store = 192;   // 180 features + 12 zero columns (zero weights / bias) per view
        if (v == 0) {        // m = y, lines = x (slab), planes = z
          p.A = a5[0] + (int64_t)ix0 * p.a_ys; p.M = by; p.Y = nx; p.Z = bz;
          p.ldc = (int64_t)bz * kFeatLd; p.c_ys = plane * kFeatLd; p.c_zs = kFeatLd;
        } else if (v == 1) { // m = z, lines = x (slab), planes = y
          p.A = a5[1] + (int64_t)ix0 * p.a_ys; p.M = bz; p.Y = nx; p.Z = by;
          p.ldc = kFeatLd; p.c_ys = plane * kFeatLd; p.c_zs = (int64_t)bz * kFeatLd;
        } else {             // m = z, lines = y, planes = x (slab)
          p.A = a5[2] + (int64_t)ix0 * p.a_zs; p.M = bz; p.Y = by; p.Z = nx;
          p.ldc = kFeatLd; p.c_ys = (int64_t)bz * kFeatLd; p.c_zs = plane * kFeatLd;
        }
        p.C = feats;
        if (compact) p.rowmap = rowmap + slab_base;      // dense row -> compact feature row (or skipped)
        SC_TRY(tc ? launch_gemm_tc(ctx, p, mc ? mcw.d1[v] : ctx->br[v].d1_dense, st) : launch_gemm(ctx, p, ctx->br[v].d1_dense, st));
      }
      GemmProblem p;
      SC_CHECK(rows < (1ll << 31), SC_ERR_ARG, "sc_segment_volume: chunk too large");
      gemm_problem_rows(p, feats, kFeatLd, kFeatLd, (int)rows_fc);
      p.C = h1; p.ldc = kH1Ld; p.n_store = 540; p.out_split = tc ? 1 : 0;
      p.prof_cls = PC_GEMM_FC1;
      const bool atlas_fused = tc;   // the CTA-pair kernel writes the atlas columns in its epilogue
      if (ctx->atlas_ready && ctx->atlas_chunks == 0) {   // an atlas upload on a side stream (sc_atlas_ready_event): the priors are first
        SC_CUDA(cudaStreamWaitEvent(st, ctx->atlas_ready, 0));   // read here, after the conv phase and the first slab's d1 launches
        ctx->atlas_ready = nullptr;
      }
      if (atlas_fused) { p.atlas = atlas; p.ageo = og; p.ageo.x0 = b[0] + ix0; if (compact) p.rowvox = rowvox + slab_base; }
      SC_TRY(tc ? launch_gemm_tc(ctx, p, mc ? mcw.fc1 : ctx->fc1, st) : launch_gemm(ctx, p, ctx->fc1, st));
      p.atlas = nullptr; p.rowvox = nullptr;
      if (!atlas_fused) {  // after FC1: the tensor-core epilogue writes whole 16-column chunks (columns 540..543 as zeros)
        ProfScope prof(ctx, PC_ATLAS, st);
        dense_atlas_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(atlas, og, ix0, rows, h1, tc ? 1 : 0);
        ctx->launches++;
      }
      SC_CUDA(cudaGetLastError());
      gemm_problem_rows(p, h1, kH1Ld, kH1Ld, (int)rows_fc);
      p.prof_cls = PC_GEMM_FC2;
      OutGeo og2 = og;
      og2.x0 = b[0] + ix0;
      if (tc) {   // fc_2 with the out_layer, softmax / argmax and the scatter into the volume in its epilogue
        SoftmaxOut smo = {proba_vol, nullptr, label_vol, cand, og2, 1, compact ? rowvox + slab_base : nullptr};
        p.C = nullptr; p.ldc = 0; p.n_store = kH2Ld; p.sm = &smo;
        if (mc) { p.mc_acc = mc_acc; p.mc_first = pass == 0; }   // one Monte-Carlo pass: accumulate instead of the scatter
        SC_TRY(launch_gemm_tc(ctx, p, mc ? mcw.fc2 : ctx->fc2, st));
      } else {
        p.C = h2; p.ldc = kH2Ld; p.n_store = kH2Ld;
        SC_TRY(launch_gemm(ctx, p, ctx->fc2, st));
        SC_TRY(launch_out_softmax(ctx, h2, rows, proba_vol, nullptr, label_vol, cand, &og2, st));
      }
    }
    if (mc) {
      OutGeo og3 = og;
      og3.x0 = b[0] + ix0;
      SC_TRY(launch_mc_finalize(ctx, mc_acc, rows_fc, mc->samples, compact ? rowvox + slab_base : nullptr, og3, cand, label_vol,
                                proba_vol, mc->entropy, mc->mi, st));
    }
  }
  if (ctx->atlas_ready && ctx->atlas_chunks == 0) {     // no slab had a candidate: still join the upload before the caller goes on
    SC_CUDA(cudaStreamWaitEvent(st, ctx->atlas_ready, 0));
    ctx->atlas_ready = nullptr;
  }
  return SC_OK;
}

}  // namespace sc
