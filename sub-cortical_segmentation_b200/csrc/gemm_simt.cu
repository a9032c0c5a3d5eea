// fp32 SIMT back-end of the dense-layer / implicit-GEMM problem (exact fp32 products).
// It is the bring-up and cross-check path for gemm_tc.cu (tcgen05) and the only path for
// the 270->15 output layer + softmax (+argmax), which is too narrow for a tensor-core tile.
//
// Reference ops replaced: DenseLayer + PReLU at cnn_cort/nets.py:179-180,217-218,227-228 and
// DenseLayer(softmax) at :231; nolearn predict = argmax(predict_proba) (first maximum wins).
#include "common.cuh"

namespace sc {

constexpr int BM = 128, BN = 64, BK = 16;
constexpr int AS_LD = BM + 4;

struct GemmArgs {
  GemmProblem p;
  const float* W;  // [Kpad][Npad]
  const float* bias;
  const float* alpha;
  int Npad;
  int mt, nt;
};

__global__ void __launch_bounds__(256) gemm_simt_kernel(const GemmArgs a) {
  __shared__ __align__(16) float As[BK][AS_LD];
  __shared__ __align__(16) float Bs[BK][BN];
  const GemmProblem& p = a.p;
  int64_t bid = blockIdx.x;
  const int n_tile = (int)(bid % a.nt); bid /= a.nt;
  const int m_tile = (int)(bid % a.mt); bid /= a.mt;
  const int y = (int)(bid % p.Y);
  const int z = (int)(bid / p.Y);
  const int m0 = m_tile * BM, n0 = n_tile * BN;
  const float* Abase = p.A + (int64_t)z * p.a_zs + (int64_t)y * p.a_ys;
  const int tid = threadIdx.x, tm = tid & 15, tn = tid >> 4;

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int tap = 0; tap < p.ntaps; ++tap) {
    const float* At = Abase + p.tap_off[tap];
    const float* Wt = a.W + (int64_t)tap * p.kc * a.Npad;
    for (int k0 = 0; k0 < p.kc; k0 += BK) {
      // A tile: 128 rows x 16 k -> transposed into As[k][m]
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int idx = tid + r * 256, row = idx >> 2, kq = idx & 3;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m0 + row < p.M) v = __ldg(reinterpret_cast<const float4*>(At + (int64_t)(m0 + row) * p.lda + k0 + kq * 4));
        As[kq * 4 + 0][row] = v.x; As[kq * 4 + 1][row] = v.y; As[kq * 4 + 2][row] = v.z; As[kq * 4 + 3][row] = v.w;
      }
      {  // B tile: 16 k x 64 n
        const int kr = tid >> 4, nq = tid & 15;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n0 + nq * 4 < a.Npad) v = __ldg(reinterpret_cast<const float4*>(Wt + (int64_t)(k0 + kr) * a.Npad + n0 + nq * 4));
        *reinterpret_cast<float4*>(&Bs[kr][nq * 4]) = v;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        const float4 a0 = *reinterpret_cast<const float4*>(&As[k][tm * 8]);
        const float4 a1 = *reinterpret_cast<const float4*>(&As[k][tm * 8 + 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tn * 4]);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  const int n = n0 + tn * 4;
  if (n >= p.n_store) return;
  const float4 bias = __ldg(reinterpret_cast<const float4*>(a.bias + n));
  const float4 al = __ldg(reinterpret_cast<const float4*>(a.alpha + n));
  float* Cbase = p.C + (int64_t)z * p.c_zs + (int64_t)y * p.c_ys;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + tm * 8 + i;
    if (m >= p.M) break;
    float4 v;
    v.x = prelu(acc[i][0] + bias.x, al.x);
    v.y = prelu(acc[i][1] + bias.y, al.y);
    v.z = prelu(acc[i][2] + bias.z, al.z);
    v.w = prelu(acc[i][3] + bias.w, al.w);
    *reinterpret_cast<float4*>(Cbase + (int64_t)m * p.ldc + p.c_col0 + n) = v;
  }
}

int launch_gemm(sc_ctx* ctx, const GemmProblem& p, const GemmW& w, cudaStream_t st) {
  if (p.M <= 0 || p.Y <= 0 || p.Z <= 0) return SC_OK;
  SC_CHECK(p.kc % BK == 0 && p.n_store % 4 == 0 && p.n_store <= w.Npad, SC_ERR_ARG, "gemm: bad geometry kc=%d n_store=%d", p.kc, p.n_store);
  SC_CHECK(p.ntaps * p.kc == w.Kpad, SC_ERR_ARG, "gemm: K mismatch %d*%d vs %d", p.ntaps, p.kc, w.Kpad);
  SC_CHECK(!p.out_split && p.c_col0 % 4 == 0, SC_ERR_ARG, "gemm: the SIMT back-end writes plain fp32 rows only");
  GemmArgs a;
  a.p = p; a.W = w.w_kn; a.bias = w.bias; a.alpha = w.alpha; a.Npad = w.Npad;
  a.mt = (p.M + BM - 1) / BM;
  a.nt = (p.n_store + BN - 1) / BN;
  const int64_t blocks = (int64_t)a.mt * a.nt * p.Y * p.Z;
  SC_CHECK(blocks < (1ll << 31), SC_ERR_ARG, "gemm: grid too large");
  ProfScope prof(ctx, p.prof_cls, st);
  gemm_simt_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// out_layer (270 -> 15) + softmax + argmax of the SIMT back-end (the tcgen05 back-end fuses them into fc_2): one thread per voxel (each thread streams its own 1 088 B row
// through L1 with float4 loads; the 16 KB weight matrix is read from shared memory as warp-wide broadcasts).
__global__ void __launch_bounds__(128) out_softmax_kernel(const float* __restrict__ h2, int64_t n,
                                                          const float* __restrict__ W, const float* __restrict__ b,
                                                          float* __restrict__ proba, int32_t* __restrict__ label,
                                                          uint8_t* __restrict__ label8, const uint8_t* __restrict__ mask,
                                                          const OutGeo geo, const int use_geo) {
  __shared__ __align__(16) float sW[270 * 16];
  for (int i = threadIdx.x; i < 270 * 16; i += 128) sW[i] = W[i];
  __syncthreads();
  const int64_t v = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (v >= n) return;
  int64_t o = v;
  if (use_geo) {
    const int64_t plane = (int64_t)geo.by * geo.bz;
    const int ix = (int)(v / plane);
    const int rem = (int)(v - (int64_t)ix * plane);
    const int iy = rem / geo.bz, iz = rem - iy * geo.bz;
    o = ((int64_t)(geo.x0 + ix) * geo.Y + (geo.y0 + iy)) * geo.Z + (geo.z0 + iz);
    if (mask && mask[o] == 0) return;
  }
  const float4* row = reinterpret_cast<const float4*>(h2 + v * kH2Ld);
  float z[15];
#pragma unroll
  for (int c = 0; c < 15; ++c) z[c] = __ldg(b + c);
#pragma unroll 2
  for (int k4 = 0; k4 < 68; ++k4) {
    const float4 xv = __ldg(row + k4);
    const float x[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k4 * 4 + j;
      if (k < 270) {
        const float4* w4 = reinterpret_cast<const float4*>(sW + k * 16);
        const float4 w0 = w4[0], w1 = w4[1], w2 = w4[2], w3 = w4[3];
        z[0] = fmaf(x[j], w0.x, z[0]); z[1] = fmaf(x[j], w0.y, z[1]); z[2] = fmaf(x[j], w0.z, z[2]); z[3] = fmaf(x[j], w0.w, z[3]);
        z[4] = fmaf(x[j], w1.x, z[4]); z[5] = fmaf(x[j], w1.y, z[5]); z[6] = fmaf(x[j], w1.z, z[6]); z[7] = fmaf(x[j], w1.w, z[7]);
        z[8] = fmaf(x[j], w2.x, z[8]); z[9] = fmaf(x[j], w2.y, z[9]); z[10] = fmaf(x[j], w2.z, z[10]); z[11] = fmaf(x[j], w2.w, z[11]);
        z[12] = fmaf(x[j], w3.x, z[12]); z[13] = fmaf(x[j], w3.y, z[13]); z[14] = fmaf(x[j], w3.z, z[14]);
      }
    }
  }
  softmax_store(z, o, proba, label, label8);
}

int launch_out_softmax(sc_ctx* ctx, const float* h2, int64_t n, float* proba, int32_t* label, uint8_t* label8,
                       const uint8_t* mask, const OutGeo* geo, cudaStream_t st) {
  if (n == 0) return SC_OK;
  const int64_t blocks = (n + 127) / 128;
  SC_CHECK(blocks < (1ll << 31), SC_ERR_ARG, "out_softmax: too many rows");
  const unsigned grid = (unsigned)blocks;
  OutGeo g = geo ? *geo : OutGeo{0, 0, 0, 1, 1, 1, 1};
  ProfScope prof(ctx, PC_OUT, st);
  out_softmax_kernel<<<grid, 128, 0, st>>>(h2, n, ctx->out_w, ctx->out_b, proba, label, label8, mask, g, geo ? 1 : 0);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
