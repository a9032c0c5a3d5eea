// Atlas registration on the device (sc_register_affine / sc_register_ffd / sc_warp_volume / sc_register_objective /
// sc_prior_mask): the template T1 (floating) is mapped onto the subject T1 (reference) by phi(x) = A [x; 1] + u(v), an
// affine stage and a cubic B-spline free-form deformation, both ascending normalised mutual information.  Conventions and
// definitions are those of include/subcort_b200.h and oracle/register.py, which restates every step in float64.
//
//   pyramid      down_kernel: [1/4, 1/2, 1/4] per axis (edge repeated), every second voxel
//   objective    hist_kernel: one thread per (x, y) line of the subject walks z; warp (affine + B-spline field, the field
//                contracted over x and y once per control-point row and slid along z), trilinear sample, 4 x 4 Parzen
//                window products in 2^-24 fixed point into a per-CTA shared histogram, integer atomics into the global one
//                (integer sums do not depend on the order: the histogram is the same on every run).  nmi_kernel: entropies,
//                NMI and the gradient table T(r, f) = (NMI log p - log p_F) / H_RF.
//   gradient     grad_kernel: the same walk; dNMI/dF(x) = -(1/N) sum T beta3(a - r) beta3'(b - f) * bin scale, times the
//                template gradient in mm -> per-thread affine sums (double) reduced by a fixed tree, and the z pass of the
//                B-spline adjoint (each control point of the line summed by its one thread, in z order); then the y pass
//                and the x pass (one thread per output, fixed order), the latter combined with the bending-energy gradient.
//   optimiser    host loops of Polak-Ribiere conjugate directions with a backtracking step; every trial reads a few bytes
//                back (cudaMemcpyAsync into pinned memory).  All floating-point reductions are fixed-order trees in double,
//                so the same inputs give byte-identical A, grid and priors on every run.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace sc {

constexpr int kBins = 64;
constexpr int kSpacing = 5;                 // control-point spacing in voxels of each level's subject image
constexpr double kLambda = 0.001;           // bending-energy weight of the FFD objective
constexpr int kMinLevelDim = 16;            // a pyramid level is used only when both images have every dim >= this
constexpr int kAffLevels = 4, kAffIters = 50;
constexpr double kAffAlpha0 = 1.0, kAffAlphaMax = 4.0;   // level voxels: largest move of a corner of the mask's box
constexpr int kFfdLevels = 3, kFfdIters = 150;
constexpr double kFfdAlpha0 = 0.5, kFfdAlphaMax = 2.0;   // level voxels: largest control-point move
constexpr double kAlphaMin = 0.01;
constexpr float kFix = 16777216.f;          // 2^24: fixed-point unit of one Parzen product
constexpr int kLineThreads = 128;
constexpr int kRedBlocks = 256;

struct Geo {
  const float* ref; const float* flo;
  int rX, rY, rZ, fX, fY, fZ;
  float P[12];       // subject voxel -> template voxel (affine part of phi)
  float Q[9];        // template voxels per mm (inverse of the template's linear part)
  float M[12];       // subject voxel -> subject mm minus the centre c (affine gradient sums)
  float rmin, rs, fmin, fs;   // bin = 2 + (v - min) * scale
  const float* grid; int gx, gy, gz;   // grid == nullptr: affine only
};

__device__ __forceinline__ void bsw(float f, float* w) {
  const float f2 = f * f, f3 = f2 * f;
  w[0] = (1.f - f) * (1.f - f) * (1.f - f) * (1.f / 6.f);
  w[1] = (3.f * f3 - 6.f * f2 + 4.f) * (1.f / 6.f);
  w[2] = (-3.f * f3 + 3.f * f2 + 3.f * f + 1.f) * (1.f / 6.f);
  w[3] = f3 * (1.f / 6.f);
}

__device__ __forceinline__ float parzen(float t) {
  const float a = fabsf(t);
  return a < 1.f ? 2.f / 3.f - a * a + 0.5f * a * a * a : (a < 2.f ? (2.f - a) * (2.f - a) * (2.f - a) * (1.f / 6.f) : 0.f);
}
__device__ __forceinline__ float dparzen(float t) {
  const float a = fabsf(t);
  return a < 1.f ? -2.f * t + 1.5f * t * a : (a < 2.f ? -0.5f * copysignf(1.f, t) * (2.f - a) * (2.f - a) : 0.f);
}

// trilinear value and voxel gradient of a [X][Y][Z] volume; false outside [0, d-1]^3
__device__ __forceinline__ bool sample(const float* __restrict__ v, int X, int Y, int Z, float wx, float wy, float wz, float& val,
                                       float* g) {
  if (!(wx >= 0.f && wy >= 0.f && wz >= 0.f && wx <= X - 1 && wy <= Y - 1 && wz <= Z - 1)) return false;
  const int i = min((int)wx, X - 2), j = min((int)wy, Y - 2), k = min((int)wz, Z - 2);
  const float fx = wx - i, fy = wy - j, fz = wz - k;
  const float* p = v + ((size_t)i * Y + j) * Z + k;
  const size_t sx = (size_t)Y * Z;
  const float c000 = __ldg(p), c001 = __ldg(p + 1), c010 = __ldg(p + Z), c011 = __ldg(p + Z + 1);
  const float c100 = __ldg(p + sx), c101 = __ldg(p + sx + 1), c110 = __ldg(p + sx + Z), c111 = __ldg(p + sx + Z + 1);
  const float c00 = c000 + fz * (c001 - c000), c01 = c010 + fz * (c011 - c010);
  const float c10 = c100 + fz * (c101 - c100), c11 = c110 + fz * (c111 - c110);
  const float c0 = c00 + fy * (c01 - c00), c1 = c10 + fy * (c11 - c10);
  val = c0 + fx * (c1 - c0);
  if (g) {
    g[0] = c1 - c0;
    g[1] = (1.f - fx) * (c01 - c00) + fx * (c11 - c10);
    const float d00 = c001 - c000, d01 = c011 - c010, d10 = c101 - c100, d11 = c111 - c110;
    g[2] = (1.f - fx) * ((1.f - fy) * d00 + fy * d01) + fx * ((1.f - fy) * d10 + fy * d11);
  }
  return true;
}

// sum over the 4 x 4 control points of the line's (x, y) cell at grid z index k
__device__ __forceinline__ float3 contract(const Geo& g, int ix0, int iy0, const float* wx, const float* wy, int k) {
  float3 u = make_float3(0.f, 0.f, 0.f);
  for (int a = 0; a < 4; ++a)
    for (int b = 0; b < 4; ++b) {
      const float w = wx[a] * wy[b];
      const float* c = g.grid + (((size_t)(ix0 + a) * g.gy + iy0 + b) * g.gz + k) * 3;
      u.x += w * __ldg(c); u.y += w * __ldg(c + 1); u.z += w * __ldg(c + 2);
    }
  return u;
}

// One subject line: calls visit(z, r, w[3], wz[4]) for every masked voxel whose image lies inside the template, and
// emit(k) when grid z index k can receive no further contribution (every k exactly once, in increasing order).
template <class Visit, class Emit>
__device__ __forceinline__ void walk_line(const Geo& g, int x, int y, Visit visit, Emit emit) {
  const float* rrow = g.ref + ((size_t)x * g.rY + y) * g.rZ;
  const float bx = g.P[0] * x + g.P[1] * y + g.P[3], by = g.P[4] * x + g.P[5] * y + g.P[7], bz = g.P[8] * x + g.P[9] * y + g.P[11];
  const bool ffd = g.grid != nullptr;
  float wxs[4], wys[4], wzs[4] = {0.f, 0.f, 0.f, 0.f};
  int ix0 = 0, iy0 = 0, kz = -1;
  float3 U[4];
  if (ffd) {
    ix0 = x / kSpacing; iy0 = y / kSpacing;
    bsw((x - ix0 * kSpacing) * (1.f / kSpacing), wxs);
    bsw((y - iy0 * kSpacing) * (1.f / kSpacing), wys);
  }
  for (int z = 0; z < g.rZ; ++z) {
    float ux = 0.f, uy = 0.f, uz = 0.f;
    if (ffd) {
      const int a = z / kSpacing;
      if (a != kz) {
        if (kz < 0) {
          for (int k = 0; k < 4; ++k) U[k] = contract(g, ix0, iy0, wxs, wys, a + k);
        } else {
          emit(kz);
          U[0] = U[1]; U[1] = U[2]; U[2] = U[3];
          U[3] = contract(g, ix0, iy0, wxs, wys, a + 3);
        }
        kz = a;
      }
      bsw((z - a * kSpacing) * (1.f / kSpacing), wzs);
      ux = wzs[0] * U[0].x + wzs[1] * U[1].x + wzs[2] * U[2].x + wzs[3] * U[3].x;
      uy = wzs[0] * U[0].y + wzs[1] * U[1].y + wzs[2] * U[2].y + wzs[3] * U[3].y;
      uz = wzs[0] * U[0].z + wzs[1] * U[1].z + wzs[2] * U[2].z + wzs[3] * U[3].z;
    }
    const float r = __ldg(rrow + z);
    if (r == 0.f) continue;
    float w[3];
    w[0] = bx + g.P[2] * z + g.Q[0] * ux + g.Q[1] * uy + g.Q[2] * uz;
    w[1] = by + g.P[6] * z + g.Q[3] * ux + g.Q[4] * uy + g.Q[5] * uz;
    w[2] = bz + g.P[10] * z + g.Q[6] * ux + g.Q[7] * uy + g.Q[8] * uz;
    visit(z, r, w, wzs);
  }
  if (ffd)
    for (int k = 0; k < 4; ++k) emit(kz + k);
}

__global__ void __launch_bounds__(kLineThreads) hist_kernel(Geo g, unsigned long long* __restrict__ hist, unsigned long long* __restrict__ count) {
  __shared__ unsigned long long s_h[kBins * kBins];
  __shared__ unsigned s_n;
  for (int i = threadIdx.x; i < kBins * kBins; i += blockDim.x) s_h[i] = 0;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const int line = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned n = 0;
  if (line < g.rX * g.rY) {
    walk_line(g, line / g.rY, line % g.rY, [&](int, float r, const float* w, const float*) {
      float F;
      if (!sample(g.flo, g.fX, g.fY, g.fZ, w[0], w[1], w[2], F, nullptr)) return;
      const float rb = 2.f + (r - g.rmin) * g.rs, fb = 2.f + (F - g.fmin) * g.fs;
      const int ra = (int)floorf(rb), fa = (int)floorf(fb);
      float wr[4], wf[4];
      for (int i = 0; i < 4; ++i) { wr[i] = parzen(ra + i - 1 - rb); wf[i] = parzen(fa + i - 1 - fb); }
      for (int i = 0; i < 4; ++i)
        for (int k = 0; k < 4; ++k)
          atomicAdd(&s_h[(ra + i - 1) * kBins + fa + k - 1], (unsigned long long)__float2ull_rn(wr[i] * wf[k] * kFix));
      ++n;
    }, [](int) {});
  }
  atomicAdd(&s_n, n);
  __syncthreads();
  for (int i = threadIdx.x; i < kBins * kBins; i += blockDim.x)
    if (s_h[i]) atomicAdd(&hist[i], s_h[i]);
  if (threadIdx.x == 0 && s_n) atomicAdd(count, (unsigned long long)s_n);
}

// one block of 256 threads: stat = {NMI, N, H_R, H_F, H_RF}, T = the gradient table
__global__ void __launch_bounds__(256) nmi_kernel(const unsigned long long* __restrict__ hist, const unsigned long long* __restrict__ count,
                                                   double* __restrict__ stat, float* __restrict__ T) {
  __shared__ double s_p[kBins * kBins];
  __shared__ double s_pr[kBins], s_pf[kBins];
  __shared__ double s_red[256];
  const int t = threadIdx.x;
  const double n = (double)*count;
  const double inv = n > 0 ? 1.0 / ((double)kFix * n) : 0.0;
  for (int i = t; i < kBins * kBins; i += 256) s_p[i] = (double)hist[i] * inv;
  __syncthreads();
  if (t < kBins) {
    double a = 0.0, b = 0.0;
    for (int k = 0; k < kBins; ++k) { a += s_p[t * kBins + k]; b += s_p[k * kBins + t]; }
    s_pr[t] = a; s_pf[t] = b;
  }
  double h = 0.0;
  for (int i = t; i < kBins * kBins; i += 256) h -= s_p[i] > 0 ? s_p[i] * log(s_p[i]) : 0.0;
  s_red[t] = h;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (t < s) s_red[t] += s_red[t + s];
    __syncthreads();
  }
  __shared__ double s_nmi, s_hrf;
  if (t == 0) {
    double hr = 0.0, hf = 0.0;
    for (int k = 0; k < kBins; ++k) {
      hr -= s_pr[k] > 0 ? s_pr[k] * log(s_pr[k]) : 0.0;
      hf -= s_pf[k] > 0 ? s_pf[k] * log(s_pf[k]) : 0.0;
    }
    const double hrf = s_red[0];
    s_nmi = hrf > 0 ? (hr + hf) / hrf : 0.0;
    s_hrf = hrf;
    stat[0] = s_nmi; stat[1] = n; stat[2] = hr; stat[3] = hf; stat[4] = hrf;
  }
  __syncthreads();
  for (int i = t; i < kBins * kBins; i += 256) {
    const double p = s_p[i];
    T[i] = p > 0 && s_hrf > 0 ? (float)((s_nmi * log(p) - log(s_pf[i % kBins])) / s_hrf) : 0.f;
  }
}

// gradient walk: affine sums (part[block][12], centred mm) and / or the z pass of the adjoint (gzb[line][gz][3])
__global__ void __launch_bounds__(kLineThreads) grad_kernel(Geo g, const float* __restrict__ T, const double* __restrict__ stat,
                                                            double* __restrict__ part, float* __restrict__ gzb) {
  __shared__ float s_T[kBins * kBins];
  __shared__ double s_red[kLineThreads];
  for (int i = threadIdx.x; i < kBins * kBins; i += blockDim.x) s_T[i] = T[i];
  __syncthreads();
  const float scale = (float)(-(double)g.fs / stat[1]);
  const int line = blockIdx.x * blockDim.x + threadIdx.x;
  double acc[12];
  for (int i = 0; i < 12; ++i) acc[i] = 0.0;
  if (line < g.rX * g.rY) {
    const int x = line / g.rY, y = line % g.rY;
    double cz[4][3];
    for (int k = 0; k < 4; ++k) cz[k][0] = cz[k][1] = cz[k][2] = 0.0;
    float* out = gzb ? gzb + (size_t)line * g.gz * 3 : nullptr;
    walk_line(g, x, y, [&](int z, float r, const float* w, const float* wz) {
      float F, gv[3];
      if (!sample(g.flo, g.fX, g.fY, g.fZ, w[0], w[1], w[2], F, gv)) return;
      const float rb = 2.f + (r - g.rmin) * g.rs, fb = 2.f + (F - g.fmin) * g.fs;
      const int ra = (int)floorf(rb), fa = (int)floorf(fb);
      float wr[4], wf[4];
      for (int i = 0; i < 4; ++i) { wr[i] = parzen(ra + i - 1 - rb); wf[i] = dparzen(fa + i - 1 - fb); }
      float s = 0.f;
      for (int i = 0; i < 4; ++i) {
        const float* Tr = s_T + (ra + i - 1) * kBins + fa - 1;
        s += wr[i] * (Tr[0] * wf[0] + Tr[1] * wf[1] + Tr[2] * wf[2] + Tr[3] * wf[3]);
      }
      const float dF = s * scale;
      float gm[3];   // d NMI / d phi(x) in mm: Q^T grad_vox
      for (int j = 0; j < 3; ++j) gm[j] = dF * (g.Q[j] * gv[0] + g.Q[3 + j] * gv[1] + g.Q[6 + j] * gv[2]);
      if (part) {
        float xm[3];
        for (int j = 0; j < 3; ++j) xm[j] = g.M[4 * j] * x + g.M[4 * j + 1] * y + g.M[4 * j + 2] * z + g.M[4 * j + 3];
        for (int i = 0; i < 3; ++i) {
          for (int j = 0; j < 3; ++j) acc[4 * i + j] += (double)(gm[i] * xm[j]);
          acc[4 * i + 3] += (double)gm[i];
        }
      }
      if (out)
        for (int k = 0; k < 4; ++k)
          for (int c = 0; c < 3; ++c) cz[k][c] += (double)(wz[k] * gm[c]);
    }, [&](int k) {
      if (!out) return;
      for (int c = 0; c < 3; ++c) out[(size_t)k * 3 + c] = (float)cz[0][c];
      for (int q = 0; q < 3; ++q)
        for (int c = 0; c < 3; ++c) cz[q][c] = cz[q + 1][c];
      cz[3][0] = cz[3][1] = cz[3][2] = 0.0;
    });
  }
  if (!part) return;
  for (int i = 0; i < 12; ++i) {
    s_red[threadIdx.x] = acc[i];
    __syncthreads();
    for (int s = kLineThreads / 2; s > 0; s >>= 1) {
      if (threadIdx.x < s) s_red[threadIdx.x] += s_red[threadIdx.x + s];
      __syncthreads();
    }
    if (threadIdx.x == 0) part[(size_t)blockIdx.x * 12 + i] = s_red[0];
    __syncthreads();
  }
}

// weight of control point i at voxel v (0 outside its support of 4 spacings)
__device__ __forceinline__ float bweight(int i, int v) {
  const int a = v / kSpacing, k = i - a;
  if (k < 0 || k > 3) return 0.f;
  const float f = (v - a * kSpacing) * (1.f / kSpacing), f2 = f * f, f3 = f2 * f;
  return k == 0 ? (1.f - f) * (1.f - f) * (1.f - f) * (1.f / 6.f)
       : k == 1 ? (3.f * f3 - 6.f * f2 + 4.f) * (1.f / 6.f)
       : k == 2 ? (-3.f * f3 + 3.f * f2 + 3.f * f + 1.f) * (1.f / 6.f) : f3 * (1.f / 6.f);
}

// y pass: gyb[x][j][k] = sum_y beta_j(y) gzb[x][y][k]
__global__ void adj_y_kernel(const float* __restrict__ gzb, int X, int Y, int gy, int gz, float* __restrict__ gyb) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (int64_t)X * gy * gz) return;
  const int k = (int)(o % gz), j = (int)((o / gz) % gy), x = (int)(o / ((int64_t)gz * gy));
  double s0 = 0, s1 = 0, s2 = 0;
  for (int y = max(0, (j - 3) * kSpacing); y < min(Y, (j + 1) * kSpacing); ++y) {
    const float w = bweight(j, y);
    const float* p = gzb + (((size_t)x * Y + y) * gz + k) * 3;
    s0 += (double)(w * p[0]); s1 += (double)(w * p[1]); s2 += (double)(w * p[2]);
  }
  gyb[o * 3] = (float)s0; gyb[o * 3 + 1] = (float)s1; gyb[o * 3 + 2] = (float)s2;
}

// x pass, combined with the bending energy: grad[i][j][k] = (1 - lambda) sum_x beta_i(x) gyb[x][j][k] - lambda dBE
__global__ void adj_x_kernel(const float* __restrict__ gyb, int X, int gx, int gy, int gz, const float* __restrict__ gbe, float lam,
                             float* __restrict__ grad) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t jk = (int64_t)gy * gz;
  if (o >= (int64_t)gx * jk) return;
  const int i = (int)(o / jk);
  const int64_t r = o % jk;
  double s0 = 0, s1 = 0, s2 = 0;
  for (int x = max(0, (i - 3) * kSpacing); x < min(X, (i + 1) * kSpacing); ++x) {
    const float w = bweight(i, x);
    const float* p = gyb + ((size_t)x * jk + r) * 3;
    s0 += (double)(w * p[0]); s1 += (double)(w * p[1]); s2 += (double)(w * p[2]);
  }
  grad[o * 3] = (float)((1.0 - lam) * s0 - (double)lam * gbe[o * 3]);
  grad[o * 3 + 1] = (float)((1.0 - lam) * s1 - (double)lam * gbe[o * 3 + 1]);
  grad[o * 3 + 2] = (float)((1.0 - lam) * s2 - (double)lam * gbe[o * 3 + 2]);
}

// bending energy: 1-D stencils B, D1, D2 of the B-spline at a control point; the six terms xx, yy, zz, xy, xz, yz
__constant__ float c_st[3][3] = {{1.f / 6.f, 4.f / 6.f, 1.f / 6.f}, {-0.5f, 0.f, 0.5f}, {1.f, -2.f, 1.f}};
__constant__ int c_term[6][3] = {{2, 0, 0}, {0, 2, 0}, {0, 0, 2}, {1, 1, 0}, {1, 0, 1}, {0, 1, 1}};
__constant__ float c_tw[6] = {1.f, 1.f, 1.f, 2.f, 2.f, 2.f};

// per interior control point q: the 6 x 3 second derivatives D (double) and its energy e[q]
__global__ void be_terms_kernel(const float* __restrict__ grid, int gx, int gy, int gz, double* __restrict__ D, double* __restrict__ e) {
  const int nx = gx - 2, ny = gy - 2, nz = gz - 2;
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (int64_t)nx * ny * nz) return;
  const int i = (int)(q / ((int64_t)ny * nz)) + 1, j = (int)((q / nz) % ny) + 1, k = (int)(q % nz) + 1;
  double en = 0.0;
  for (int t = 0; t < 6; ++t) {
    double d[3] = {0, 0, 0};
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b)
        for (int c = 0; c < 3; ++c) {
          const double w = (double)c_st[c_term[t][0]][a] * c_st[c_term[t][1]][b] * c_st[c_term[t][2]][c];
          const float* p = grid + (((size_t)(i + a - 1) * gy + j + b - 1) * gz + k + c - 1) * 3;
          for (int m = 0; m < 3; ++m) d[m] += w * p[m];
        }
    for (int m = 0; m < 3; ++m) { D[(q * 6 + t) * 3 + m] = d[m]; en += c_tw[t] * d[m] * d[m]; }
  }
  e[q] = en;
}

__global__ void be_grad_kernel(const double* __restrict__ D, int gx, int gy, int gz, double inv_ncp, float* __restrict__ gbe) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= (int64_t)gx * gy * gz) return;
  const int i = (int)(p / ((int64_t)gy * gz)), j = (int)((p / gz) % gy), k = (int)(p % gz);
  const int nx = gx - 2, ny = gy - 2, nz = gz - 2;
  double s[3] = {0, 0, 0};
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b)
      for (int c = 0; c < 3; ++c) {
        const int qi = i - a + 1, qj = j - b + 1, qk = k - c + 1;     // q = p - (a - 1, b - 1, c - 1)
        if (qi < 1 || qj < 1 || qk < 1 || qi > nx || qj > ny || qk > nz) continue;
        const int64_t q = ((int64_t)(qi - 1) * ny + qj - 1) * nz + qk - 1;
        for (int t = 0; t < 6; ++t) {
          const double w = 2.0 * c_tw[t] * c_st[c_term[t][0]][a] * c_st[c_term[t][1]][b] * c_st[c_term[t][2]][c];
          for (int m = 0; m < 3; ++m) s[m] += w * D[(q * 6 + t) * 3 + m];
        }
      }
  for (int m = 0; m < 3; ++m) gbe[p * 3 + m] = (float)(s[m] * inv_ncp);
}

// fixed-order reductions: per-block partials (grid-stride in a fixed pattern, then a shared-memory tree) and one block
// that folds the partials of every column.  mode 0: sum a*a | sum a*b (2 columns); 1: max |a_cp| over 3-vectors; 2: sum a
__global__ void __launch_bounds__(256) vec_part_kernel(const float* __restrict__ a, const float* __restrict__ b, const double* __restrict__ ad,
                                                       int64_t n, int mode, double* __restrict__ part) {
  __shared__ double s0[256], s1[256];
  double x0 = 0.0, x1 = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (mode == 0) { x0 += (double)a[i] * a[i]; x1 += (double)a[i] * b[i]; }
    else if (mode == 1) x0 = fmax(x0, sqrt((double)a[3 * i] * a[3 * i] + (double)a[3 * i + 1] * a[3 * i + 1] + (double)a[3 * i + 2] * a[3 * i + 2]));
    else x0 += ad[i];
  }
  s0[threadIdx.x] = x0; s1[threadIdx.x] = x1;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      s0[threadIdx.x] = mode == 1 ? fmax(s0[threadIdx.x], s0[threadIdx.x + s]) : s0[threadIdx.x] + s0[threadIdx.x + s];
      s1[threadIdx.x] += s1[threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { part[blockIdx.x * 2] = s0[0]; part[blockIdx.x * 2 + 1] = s1[0]; }
}

// out[c] = fold over rows of in[row][c] (cols <= 16), sum or max, in row order per thread then a tree
__global__ void __launch_bounds__(256) fold_kernel(const double* __restrict__ in, int rows, int cols, int is_max, double* __restrict__ out) {
  __shared__ double s[256];
  for (int c = 0; c < cols; ++c) {
    double x = 0.0;
    for (int r = threadIdx.x; r < rows; r += 256) x = is_max ? fmax(x, in[(size_t)r * cols + c]) : x + in[(size_t)r * cols + c];
    s[threadIdx.x] = x;
    __syncthreads();
    for (int h = 128; h > 0; h >>= 1) {
      if (threadIdx.x < h) s[threadIdx.x] = is_max ? fmax(s[threadIdx.x], s[threadIdx.x + h]) : s[threadIdx.x] + s[threadIdx.x + h];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[c] = s[0];
    __syncthreads();
  }
}

__global__ void axpy_kernel(float* __restrict__ out, const float* __restrict__ x, float a, const float* __restrict__ d, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = x[i] + a * d[i];
}

// pyramid: [1/4, 1/2, 1/4] separable smoothing with repeated edges, every second voxel
__global__ void down_kernel(const float* __restrict__ in, int X, int Y, int Z, float* __restrict__ out, int X2, int Y2, int Z2) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (int64_t)X2 * Y2 * Z2) return;
  const int x = (int)(o / ((int64_t)Y2 * Z2)), y = (int)((o / Z2) % Y2), z = (int)(o % Z2);
  const float w[3] = {0.25f, 0.5f, 0.25f};
  float s = 0.f;
  for (int a = 0; a < 3; ++a) {
    const int xi = min(max(2 * x + a - 1, 0), X - 1);
    float sy = 0.f;
    for (int b = 0; b < 3; ++b) {
      const int yi = min(max(2 * y + b - 1, 0), Y - 1);
      const float* p = in + ((size_t)xi * Y + yi) * Z;
      float sz = 0.f;
      for (int c = 0; c < 3; ++c) sz += w[c] * p[min(max(2 * z + c - 1, 0), Z - 1)];
      sy += w[b] * sz;
    }
    s += w[a] * sy;
  }
  out[o] = s;
}

__device__ __forceinline__ unsigned fkey(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float unkey(unsigned k) {
  const unsigned u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// stats[0..1] min / max keys, [2..7] box {x0, x1, y0, y1, z0, z1} (masked: only voxels != 0)
__global__ void range_kernel(const float* __restrict__ v, int X, int Y, int Z, int masked, unsigned* __restrict__ st) {
  const int64_t n = (int64_t)X * Y * Z;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float f = v[i];
    if (masked && f == 0.f) continue;
    const unsigned k = fkey(f);
    atomicMin(&st[0], k); atomicMax(&st[1], k);
    if (masked) {
      const int x = (int)(i / ((int64_t)Y * Z)), y = (int)((i / Z) % Y), z = (int)(i % Z);
      atomicMin(&st[2], (unsigned)x); atomicMax(&st[3], (unsigned)x + 1);
      atomicMin(&st[4], (unsigned)y); atomicMax(&st[5], (unsigned)y + 1);
      atomicMin(&st[6], (unsigned)z); atomicMax(&st[7], (unsigned)z + 1);
    }
  }
}

// intensity-weighted sums {sum v, sum v x_mm} per block (part[block][4])
__global__ void __launch_bounds__(256) com_kernel(const float* __restrict__ v, int X, int Y, int Z, Geo m, double* __restrict__ part) {
  __shared__ double s[4][256];
  double a[4] = {0, 0, 0, 0};
  const int64_t n = (int64_t)X * Y * Z;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double f = v[i];
    if (f == 0.0) continue;
    const int x = (int)(i / ((int64_t)Y * Z)), y = (int)((i / Z) % Y), z = (int)(i % Z);
    a[0] += f;
    for (int j = 0; j < 3; ++j) a[1 + j] += f * ((double)m.M[4 * j] * x + (double)m.M[4 * j + 1] * y + (double)m.M[4 * j + 2] * z + m.M[4 * j + 3]);
  }
  for (int j = 0; j < 4; ++j) s[j][threadIdx.x] = a[j];
  __syncthreads();
  for (int h = 128; h > 0; h >>= 1) {
    if (threadIdx.x < h)
      for (int j = 0; j < 4; ++j) s[j][threadIdx.x] += s[j][threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0)
    for (int j = 0; j < 4; ++j) part[blockIdx.x * 4 + j] = s[j][0];
}

// exact cubic B-spline refinement: fine cp j on coarse cp (j + 1) / 2 (odd j: 1/8, 6/8, 1/8) or between j / 2 and j / 2 + 1
// (even j: 1/2, 1/2), per axis
__device__ __forceinline__ int refine_taps(int j, int* idx, float* w) {
  const int i = (j + 1) / 2;
  if (j & 1) { idx[0] = i - 1; idx[1] = i; idx[2] = i + 1; w[0] = 0.125f; w[1] = 0.75f; w[2] = 0.125f; return 3; }
  idx[0] = j / 2; idx[1] = j / 2 + 1; w[0] = w[1] = 0.5f;
  return 2;
}
__global__ void subdivide_kernel(const float* __restrict__ c, int cx, int cy, int cz, float* __restrict__ f, int fx, int fy, int fz) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (int64_t)fx * fy * fz) return;
  const int i = (int)(o / ((int64_t)fy * fz)), j = (int)((o / fz) % fy), k = (int)(o % fz);
  int ia[3], ja[3], ka[3];
  float wa[3], wb[3], wc[3];
  const int na = refine_taps(i, ia, wa), nb = refine_taps(j, ja, wb), nc = refine_taps(k, ka, wc);
  double s[3] = {0, 0, 0};
  for (int a = 0; a < na; ++a)
    for (int b = 0; b < nb; ++b)
      for (int q = 0; q < nc; ++q) {
        const float* p = c + (((size_t)min(ia[a], cx - 1) * cy + min(ja[b], cy - 1)) * cz + min(ka[q], cz - 1)) * 3;
        const double w = (double)wa[a] * wb[b] * wc[q];
        for (int m = 0; m < 3; ++m) s[m] += w * p[m];
      }
  for (int m = 0; m < 3; ++m) f[o * 3 + m] = (float)s[m];
}

// warp: out[v][c] = flo(phi(v))[c] (channels-last), 0 outside; the field is summed directly over the 4^3 control points
__global__ void warp_kernel(Geo g, const float* __restrict__ flo, int C, float* __restrict__ out) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (int64_t)g.rX * g.rY * g.rZ) return;
  const int x = (int)(o / ((int64_t)g.rY * g.rZ)), y = (int)((o / g.rZ) % g.rY), z = (int)(o % g.rZ);
  float u[3] = {0.f, 0.f, 0.f};
  if (g.grid) {
    const int ix = x / kSpacing, iy = y / kSpacing, iz = z / kSpacing;
    float wx[4], wy[4], wz[4];
    bsw((x - ix * kSpacing) * (1.f / kSpacing), wx);
    bsw((y - iy * kSpacing) * (1.f / kSpacing), wy);
    bsw((z - iz * kSpacing) * (1.f / kSpacing), wz);
    for (int a = 0; a < 4; ++a)
      for (int b = 0; b < 4; ++b) {
        float t[3] = {0.f, 0.f, 0.f};
        for (int c = 0; c < 4; ++c) {
          const float* p = g.grid + (((size_t)(ix + a) * g.gy + iy + b) * g.gz + iz + c) * 3;
          for (int m = 0; m < 3; ++m) t[m] += wz[c] * __ldg(p + m);
        }
        for (int m = 0; m < 3; ++m) u[m] += wx[a] * wy[b] * t[m];
      }
  }
  float w[3];
  for (int j = 0; j < 3; ++j)
    w[j] = g.P[4 * j] * x + g.P[4 * j + 1] * y + g.P[4 * j + 2] * z + g.P[4 * j + 3] + g.Q[3 * j] * u[0] + g.Q[3 * j + 1] * u[1] + g.Q[3 * j + 2] * u[2];
  float* dst = out + o * C;
  const int X = g.fX, Y = g.fY, Z = g.fZ;
  if (!(w[0] >= 0.f && w[1] >= 0.f && w[2] >= 0.f && w[0] <= X - 1 && w[1] <= Y - 1 && w[2] <= Z - 1)) {
    for (int c = 0; c < C; ++c) dst[c] = 0.f;
    return;
  }
  const int i = min((int)w[0], X - 2), j = min((int)w[1], Y - 2), k = min((int)w[2], Z - 2);
  const float fx = w[0] - i, fy = w[1] - j, fz = w[2] - k;
  const size_t sx = (size_t)Y * Z * C, sy = (size_t)Z * C;
  const float* p = flo + (((size_t)i * Y + j) * Z + k) * C;
  for (int c = 0; c < C; ++c) {
    const float c00 = p[c] + fz * (p[C + c] - p[c]), c01 = p[sy + c] + fz * (p[sy + C + c] - p[sy + c]);
    const float c10 = p[sx + c] + fz * (p[sx + C + c] - p[sx + c]), c11 = p[sx + sy + c] + fz * (p[sx + sy + C + c] - p[sx + sy + c]);
    const float c0 = c00 + fy * (c01 - c00), c1 = c10 + fy * (c11 - c10);
    dst[c] = c0 + fx * (c1 - c0);
  }
}

__global__ void prior_any_kernel(const float* __restrict__ pr, int64_t n, uint8_t* __restrict__ m) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  uint8_t any = 0;
  for (int c = 0; c < 13; ++c) any |= pr[v * 15 + c] > 0.f;
  m[v] = any;
}
__global__ void u8_to_f32_kernel(const uint8_t* __restrict__ m, int64_t n, float* __restrict__ out) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) out[v] = m[v] ? 1.f : 0.f;
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
static inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

struct Mat { double m[16]; };
static Mat mul(const Mat& a, const Mat& b) {
  Mat c;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      double s = 0;
      for (int k = 0; k < 4; ++k) s += a.m[4 * i + k] * b.m[4 * k + j];
      c.m[4 * i + j] = s;
    }
  return c;
}
static bool inv4(const Mat& a, Mat& out) {   // affine inverse (last row 0 0 0 1)
  const double* m = a.m;
  const double det = m[0] * (m[5] * m[10] - m[6] * m[9]) - m[1] * (m[4] * m[10] - m[6] * m[8]) + m[2] * (m[4] * m[9] - m[5] * m[8]);
  if (!isfinite(det) || fabs(det) < 1e-12) return false;
  double r[9] = {(m[5] * m[10] - m[6] * m[9]) / det, (m[2] * m[9] - m[1] * m[10]) / det, (m[1] * m[6] - m[2] * m[5]) / det,
                 (m[6] * m[8] - m[4] * m[10]) / det, (m[0] * m[10] - m[2] * m[8]) / det, (m[2] * m[4] - m[0] * m[6]) / det,
                 (m[4] * m[9] - m[5] * m[8]) / det, (m[1] * m[8] - m[0] * m[9]) / det, (m[0] * m[5] - m[1] * m[4]) / det};
  memset(out.m, 0, sizeof(out.m));
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) out.m[4 * i + j] = r[3 * i + j];
    out.m[4 * i + 3] = -(r[3 * i] * m[3] + r[3 * i + 1] * m[7] + r[3 * i + 2] * m[11]);
  }
  out.m[15] = 1.0;
  return true;
}
static Mat scaled(const Mat& a, int level) {
  Mat b = a;
  const double f = (double)(1 << level);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) b.m[4 * i + j] *= f;
  return b;
}

void ffd_grid_dims(const int32_t* d, int32_t* g) {
  for (int i = 0; i < 3; ++i) g[i] = (d[i] - 1) / kSpacing + 4;
}

// one registration call: pyramids, scratch and the primitive evaluations
struct Reg {
  sc_ctx* ctx; cudaStream_t st;
  int nlev = 1;
  const float* ref[4]; const float* flo[4];
  int rd[4][3], fd[4][3];
  Mat MR[4], MF[4], MFi[4];
  unsigned long long* hist; float* T; double* stat; double* part; double* fold; unsigned* rng;
  float* gzb; float* gyb; double* beD; double* beE; float* gbe;
  float* gbuf[5];   // grid, trial, dir, g, g_new
  double* h;        // pinned host: 64 doubles
  char* arena; size_t used;

  template <class T_> T_* carve(size_t n) {
    T_* p = reinterpret_cast<T_*>(arena + used);
    used += (n * sizeof(T_) + 255) & ~(size_t)255;
    return p;
  }

  int fetch(const double* dsrc, int n) {   // the optimiser's few bytes per trial
    SC_CUDA(cudaMemcpyAsync(h, dsrc, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    SC_CUDA(cudaStreamSynchronize(st));
    return SC_OK;
  }
};

static size_t vox(const int* d) { return (size_t)d[0] * d[1] * d[2]; }

static int reg_setup(Reg& R, sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                     const double* fv, int levels, bool ffd, cudaStream_t st) {
  R.ctx = ctx; R.st = st;
  R.ref[0] = ref; R.flo[0] = flo;
  for (int i = 0; i < 3; ++i) { R.rd[0][i] = rdims[i]; R.fd[0][i] = fdims[i]; }
  memcpy(R.MR[0].m, rv, sizeof(Mat)); memcpy(R.MF[0].m, fv, sizeof(Mat));
  R.nlev = levels;
  for (int l = 1; l < levels; ++l)
    for (int i = 0; i < 3; ++i) { R.rd[l][i] = (R.rd[l - 1][i] + 1) / 2; R.fd[l][i] = (R.fd[l - 1][i] + 1) / 2; }
  for (int l = 0; l < levels; ++l) {
    R.MR[l] = scaled(R.MR[0], l); R.MF[l] = scaled(R.MF[0], l);
    if (!inv4(R.MF[l], R.MFi[l])) { set_error("internal: singular template matrix"); return SC_ERR_ARG; }
  }
  int32_t g[3];
  ffd_grid_dims(rdims, g);
  const size_t ng = (size_t)g[0] * g[1] * g[2];
  const size_t nlines = (size_t)rdims[0] * rdims[1];
  size_t bytes = 0;
  auto add = [&](size_t b) { bytes += (b + 255) & ~(size_t)255; };
  for (int l = 1; l < levels; ++l) { add(vox(R.rd[l]) * 4); add(vox(R.fd[l]) * 4); }
  add((kBins * kBins + 1) * 8); add(kBins * kBins * 4); add(16 * 8); add(nblk(nlines, kLineThreads) * 12 * 8 + kRedBlocks * 4 * 8);
  add(64 * 8); add(8 * 4);
  if (ffd) {
    add(nlines * g[2] * 12); add((size_t)rdims[0] * g[1] * g[2] * 12); add(ng * 18 * 8); add(ng * 8); add(ng * 12);
    for (int i = 0; i < 5; ++i) add(ng * 12);
  }
  SC_TRY(ensure_ws(ctx->ws_reg, bytes));
  if (!ctx->h_reg) SC_CUDA(cudaMallocHost(&ctx->h_reg, 64 * sizeof(double)));
  R.h = ctx->h_reg;
  R.arena = (char*)ctx->ws_reg.ptr; R.used = 0;
  for (int l = 1; l < levels; ++l) { R.ref[l] = R.carve<float>(vox(R.rd[l])); R.flo[l] = R.carve<float>(vox(R.fd[l])); }
  R.hist = R.carve<unsigned long long>(kBins * kBins + 1);   // histogram | voxel count
  R.T = R.carve<float>(kBins * kBins); R.stat = R.carve<double>(16);
  R.part = R.carve<double>(nblk(nlines, kLineThreads) * 12 + kRedBlocks * 4); R.fold = R.carve<double>(64); R.rng = R.carve<unsigned>(8);
  if (ffd) {
    R.gzb = R.carve<float>(nlines * g[2] * 3); R.gyb = R.carve<float>((size_t)rdims[0] * g[1] * g[2] * 3);
    R.beD = R.carve<double>(ng * 18); R.beE = R.carve<double>(ng); R.gbe = R.carve<float>(ng * 3);
    for (int i = 0; i < 5; ++i) R.gbuf[i] = R.carve<float>(ng * 3);
  }
  for (int l = 1; l < levels; ++l) {
    ProfScope ps(ctx, PC_REGISTER, st);
    down_kernel<<<nblk(vox(R.rd[l]), 256), 256, 0, st>>>(R.ref[l - 1], R.rd[l - 1][0], R.rd[l - 1][1], R.rd[l - 1][2], (float*)R.ref[l],
                                                          R.rd[l][0], R.rd[l][1], R.rd[l][2]);
    down_kernel<<<nblk(vox(R.fd[l]), 256), 256, 0, st>>>(R.flo[l - 1], R.fd[l - 1][0], R.fd[l - 1][1], R.fd[l - 1][2], (float*)R.flo[l],
                                                          R.fd[l][0], R.fd[l][1], R.fd[l][2]);
    ctx->launches += 2;
  }
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// coarsest first: level 0 and the levels at which both images have every dim >= kMinLevelDim
static int used_levels(const Reg& R, int* out) {
  int n = 0;
  for (int l = R.nlev - 1; l >= 0; --l) {
    bool ok = l == 0;
    if (!ok) {
      ok = true;
      for (int i = 0; i < 3; ++i) ok = ok && R.rd[l][i] >= kMinLevelDim && R.fd[l][i] >= kMinLevelDim;
    }
    if (ok) out[n++] = l;
  }
  return n;
}

struct LevelInfo { float rmin, rs, fmin, fs; int box[6]; };

static int level_info(Reg& R, int l, LevelInfo& L) {
  unsigned init[16] = {0xffffffffu, 0u, 0xffffffffu, 0u, 0xffffffffu, 0u, 0xffffffffu, 0u, 0xffffffffu, 0u};
  SC_CUDA(cudaMemcpyAsync(R.rng, init, 8 * sizeof(unsigned), cudaMemcpyHostToDevice, R.st));
  {
    ProfScope ps(R.ctx, PC_REGISTER, R.st);
    range_kernel<<<2 * R.ctx->sm_count, 256, 0, R.st>>>(R.ref[l], R.rd[l][0], R.rd[l][1], R.rd[l][2], 1, R.rng);
    R.ctx->launches++;
  }
  SC_CUDA(cudaGetLastError());
  unsigned h[8];
  SC_CUDA(cudaMemcpyAsync(R.h, R.rng, sizeof(h), cudaMemcpyDeviceToHost, R.st));
  SC_CUDA(cudaStreamSynchronize(R.st));
  memcpy(h, R.h, sizeof(h));
  SC_CHECK(h[1] != 0u, SC_ERR_ARG, "reference volume: the mask (voxels != 0) is empty");
  const float rmin = unkey(h[0]), rmax = unkey(h[1]);
  for (int i = 0; i < 6; ++i) L.box[i] = (int)h[2 + i];
  SC_CUDA(cudaMemcpyAsync(R.rng, init, 8 * sizeof(unsigned), cudaMemcpyHostToDevice, R.st));
  {
    ProfScope ps(R.ctx, PC_REGISTER, R.st);
    range_kernel<<<2 * R.ctx->sm_count, 256, 0, R.st>>>(R.flo[l], R.fd[l][0], R.fd[l][1], R.fd[l][2], 0, R.rng);
    R.ctx->launches++;
  }
  SC_CUDA(cudaGetLastError());
  SC_CUDA(cudaMemcpyAsync(R.h, R.rng, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, R.st));
  SC_CUDA(cudaStreamSynchronize(R.st));
  memcpy(h, R.h, 2 * sizeof(unsigned));
  const float fmin = unkey(h[0]), fmax = unkey(h[1]);
  L.rmin = rmin; L.rs = (float)(59.0 / std::max((double)rmax - rmin, 1e-30));
  L.fmin = fmin; L.fs = (float)(59.0 / std::max((double)fmax - fmin, 1e-30));
  return SC_OK;
}

static Geo make_geo(const Reg& R, int l, const LevelInfo& L, const Mat& A, const double* c, const float* grid) {
  Geo g;
  g.ref = R.ref[l]; g.flo = R.flo[l];
  for (int i = 0; i < 3; ++i) { (&g.rX)[i] = R.rd[l][i]; (&g.fX)[i] = R.fd[l][i]; }
  const Mat P = mul(R.MFi[l], mul(A, R.MR[l]));
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 4; ++j) { g.P[4 * i + j] = (float)P.m[4 * i + j]; g.M[4 * i + j] = (float)R.MR[l].m[4 * i + j]; }
    for (int j = 0; j < 3; ++j) g.Q[3 * i + j] = (float)R.MFi[l].m[4 * i + j];
    g.M[4 * i + 3] = (float)(R.MR[l].m[4 * i + 3] - (c ? c[i] : 0.0));
  }
  g.rmin = L.rmin; g.rs = L.rs; g.fmin = L.fmin; g.fs = L.fs;
  g.grid = grid;
  int32_t gd[3];
  ffd_grid_dims(R.rd[l], gd);
  g.gx = gd[0]; g.gy = gd[1]; g.gz = gd[2];
  return g;
}

// NMI of one transform (also leaves T and stat on the device for grad())
static int eval_nmi(Reg& R, const Geo& g, double& nmi) {
  SC_CUDA(cudaMemsetAsync(R.hist, 0, (kBins * kBins + 1) * 8, R.st));
  {
    ProfScope ps(R.ctx, PC_REGISTER, R.st);
    hist_kernel<<<nblk((int64_t)g.rX * g.rY, kLineThreads), kLineThreads, 0, R.st>>>(g, R.hist, R.hist + kBins * kBins);
    nmi_kernel<<<1, 256, 0, R.st>>>(R.hist, R.hist + kBins * kBins, R.stat, R.T);
    R.ctx->launches += 2;
  }
  SC_CUDA(cudaGetLastError());
  SC_TRY(R.fetch(R.stat, 2));
  SC_CHECK(R.h[1] > 0, SC_ERR_ARG, "the reference mask has no overlap with the template under the transform");
  nmi = R.h[0];
  return SC_OK;
}

// BE of a grid (leaves D on the device for the gradient)
static int eval_be(Reg& R, const float* grid, int gx, int gy, int gz, double& be) {
  const int64_t nq = (int64_t)(gx - 2) * (gy - 2) * (gz - 2);
  ProfScope ps(R.ctx, PC_REGISTER, R.st);
  be_terms_kernel<<<nblk(nq, 128), 128, 0, R.st>>>(grid, gx, gy, gz, R.beD, R.beE);
  vec_part_kernel<<<kRedBlocks, 256, 0, R.st>>>(nullptr, nullptr, R.beE, nq, 2, R.part);
  fold_kernel<<<1, 256, 0, R.st>>>(R.part, kRedBlocks, 2, 0, R.fold);
  R.ctx->launches += 3;
  SC_CUDA(cudaGetLastError());
  SC_TRY(R.fetch(R.fold, 1));
  be = R.h[0] / (double)nq;
  return SC_OK;
}

// gradients at the transform of the last eval_nmi (and eval_be): affine sums (centred at c) into ga[12] (nullable);
// grid gradient d J / d grid into gout (nullable)
static int eval_grad(Reg& R, const Geo& g, double* ga, float* gout) {
  const unsigned nb = nblk((int64_t)g.rX * g.rY, kLineThreads);
  {
    ProfScope ps(R.ctx, PC_REGISTER, R.st);
    grad_kernel<<<nb, kLineThreads, 0, R.st>>>(g, R.T, R.stat, ga ? R.part : nullptr, gout ? R.gzb : nullptr);
    R.ctx->launches++;
    if (gout) {
      const int64_t ng = (int64_t)g.gx * g.gy * g.gz;
      adj_y_kernel<<<nblk((int64_t)g.rX * g.gy * g.gz, 128), 128, 0, R.st>>>(R.gzb, g.rX, g.rY, g.gy, g.gz, R.gyb);
      be_grad_kernel<<<nblk(ng, 128), 128, 0, R.st>>>(R.beD, g.gx, g.gy, g.gz, 1.0 / ((double)(g.gx - 2) * (g.gy - 2) * (g.gz - 2)), R.gbe);
      adj_x_kernel<<<nblk(ng, 128), 128, 0, R.st>>>(R.gyb, g.rX, g.gx, g.gy, g.gz, R.gbe, (float)kLambda, gout);
      R.ctx->launches += 3;
    }
    if (ga) {
      fold_kernel<<<1, 256, 0, R.st>>>(R.part, (int)nb, 12, 0, R.fold);
      R.ctx->launches++;
    }
  }
  SC_CUDA(cudaGetLastError());
  if (ga) {
    SC_TRY(R.fetch(R.fold, 12));
    memcpy(ga, R.h, 12 * sizeof(double));
  }
  return SC_OK;
}

// {sum a.a, sum a.b} or max control-point norm of a
static int vec_reduce(Reg& R, const float* a, const float* b, int64_t ncp, int mode, double* out) {
  {
    ProfScope ps(R.ctx, PC_REGISTER, R.st);
    vec_part_kernel<<<kRedBlocks, 256, 0, R.st>>>(a, b, nullptr, mode == 1 ? ncp : ncp * 3, mode, R.part);
    fold_kernel<<<1, 256, 0, R.st>>>(R.part, kRedBlocks, 2, mode == 1, R.fold);
    R.ctx->launches += 2;
  }
  SC_CUDA(cudaGetLastError());
  SC_TRY(R.fetch(R.fold, 2));
  out[0] = R.h[0]; out[1] = R.h[1];
  return SC_OK;
}

static int axpy(Reg& R, float* out, const float* x, double a, const float* d, int64_t n) {
  ProfScope ps(R.ctx, PC_REGISTER, R.st);
  axpy_kernel<<<nblk(n, 256), 256, 0, R.st>>>(out, x, (float)a, d, n);
  R.ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

static double min_spacing(const Mat& M) {
  double s = 1e300;
  for (int j = 0; j < 3; ++j) s = std::min(s, sqrt(M.m[j] * M.m[j] + M.m[4 + j] * M.m[4 + j] + M.m[8 + j] * M.m[8 + j]));
  return s;
}

int register_affine(sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                    const double* fv, double* affine_out, cudaStream_t st) {
  Reg R;
  SC_TRY(reg_setup(R, ctx, ref, rdims, rv, flo, fdims, fv, kAffLevels, false, st));
  // initial translation: intensity centres of mass (subject over its mask; template over every voxel -- zeros add nothing)
  double com[2][4];
  for (int s = 0; s < 2; ++s) {
    Geo m{};
    const Mat& M = s ? R.MF[0] : R.MR[0];
    for (int i = 0; i < 12; ++i) m.M[i] = (float)M.m[i];
    const int* d = s ? R.fd[0] : R.rd[0];
    {
      ProfScope ps(ctx, PC_REGISTER, st);
      com_kernel<<<kRedBlocks, 256, 0, st>>>(s ? flo : ref, d[0], d[1], d[2], m, R.part);
      fold_kernel<<<1, 256, 0, st>>>(R.part, kRedBlocks, 4, 0, R.fold);
      ctx->launches += 2;
    }
    SC_CUDA(cudaGetLastError());
    SC_TRY(R.fetch(R.fold, 4));
    SC_CHECK(R.h[0] != 0.0, SC_ERR_ARG, "%s", s ? "template volume: every voxel is 0" : "reference volume: the mask (voxels != 0) is empty");
    for (int j = 0; j < 4; ++j) com[s][j] = R.h[j];
  }
  Mat A;
  memset(A.m, 0, sizeof(A.m));
  A.m[0] = A.m[5] = A.m[10] = A.m[15] = 1.0;
  for (int i = 0; i < 3; ++i) A.m[4 * i + 3] = com[1][1 + i] / com[1][0] - com[0][1 + i] / com[0][0];
  const double h0 = min_spacing(R.MR[0]);
  int lv[4];
  const int nl = used_levels(R, lv);
  for (int li = 0; li < nl; ++li) {
    const int l = lv[li];
    LevelInfo L;
    SC_TRY(level_info(R, l, L));
    // box corners in mm, centre c and R^2 (oracle/register.py affine_frame)
    double corners[8][3], c[3] = {0, 0, 0};
    for (int q = 0; q < 8; ++q) {
      const double v[3] = {(double)((q & 4) ? L.box[1] - 1 : L.box[0]), (double)((q & 2) ? L.box[3] - 1 : L.box[2]),
                           (double)((q & 1) ? L.box[5] - 1 : L.box[4])};
      for (int i = 0; i < 3; ++i) {
        const double* m = R.MR[l].m + 4 * i;
        corners[q][i] = m[0] * v[0] + m[1] * v[1] + m[2] * v[2] + m[3];
        c[i] += corners[q][i] / 8.0;
      }
    }
    double R2 = 0;
    for (int q = 0; q < 8; ++q)
      for (int i = 0; i < 3; ++i) R2 += (corners[q][i] - c[i]) * (corners[q][i] - c[i]) / 24.0;
    const double Rr = sqrt(std::max(R2, 1e-12));
    auto to_A = [&](const double* th) {
      Mat B;
      memset(B.m, 0, sizeof(B.m));
      B.m[15] = 1.0;
      for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) B.m[4 * i + j] = th[3 * i + j] / Rr;
        B.m[4 * i + 3] = th[9 + i] - (B.m[4 * i] * c[0] + B.m[4 * i + 1] * c[1] + B.m[4 * i + 2] * c[2]);
      }
      return B;
    };
    auto value = [&](const double* th, double& v) -> int { return eval_nmi(R, make_geo(R, l, L, to_A(th), c, nullptr), v); };
    auto grad = [&](const double* th, double* gth) -> int {
      double G[12];
      SC_TRY(eval_grad(R, make_geo(R, l, L, to_A(th), c, nullptr), G, nullptr));
      // the sums are centred (x - c): they are already the gradient w.r.t. (L, t' = L c + t)
      for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) gth[3 * i + j] = G[4 * i + j] / Rr;
        gth[9 + i] = G[4 * i + 3];
      }
      return SC_OK;
    };
    auto norm = [&](const double* d) {
      double mx = 0;
      for (int q = 0; q < 8; ++q) {
        double s = 0;
        for (int i = 0; i < 3; ++i) {
          double m = d[9 + i];
          for (int j = 0; j < 3; ++j) m += d[3 * i + j] / Rr * (corners[q][j] - c[j]);
          s += m * m;
        }
        mx = std::max(mx, sqrt(s));
      }
      return mx;
    };
    double th[12], g[12], d[12], xt[12], gn[12];
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) th[3 * i + j] = A.m[4 * i + j] * Rr;
      th[9 + i] = A.m[4 * i] * c[0] + A.m[4 * i + 1] * c[1] + A.m[4 * i + 2] * c[2] + A.m[4 * i + 3];
    }
    const double h = h0 * (double)(1 << l);
    double J, alpha = kAffAlpha0 * h;
    SC_TRY(value(th, J));
    SC_TRY(grad(th, g));
    memcpy(d, g, sizeof(d));
    int it = 0;
    while (it < kAffIters && alpha >= kAlphaMin * h) {
      const double n = norm(d);
      if (!(n > 0)) break;
      for (int i = 0; i < 12; ++i) xt[i] = th[i] + alpha / n * d[i];
      double Jt;
      SC_TRY(value(xt, Jt));
      if (Jt > J) {
        memcpy(th, xt, sizeof(th));
        J = Jt; ++it;
        alpha = std::min(1.5 * alpha, kAffAlphaMax * h);
        SC_TRY(grad(th, gn));
        double gg = 0, num = 0;
        for (int i = 0; i < 12; ++i) { gg += g[i] * g[i]; num += gn[i] * (gn[i] - g[i]); }
        const double beta = gg > 0 ? std::max(0.0, num / gg) : 0.0;
        for (int i = 0; i < 12; ++i) { d[i] = gn[i] + beta * d[i]; g[i] = gn[i]; }
      } else {
        alpha *= 0.5;
      }
    }
    A = to_A(th);
    ctx->reg_iters[l] = it;
  }
  memcpy(affine_out, A.m, sizeof(A.m));
  return SC_OK;
}

int register_ffd(sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                 const double* fv, const double* affine, float* grid_out, cudaStream_t st) {
  Reg R;
  SC_TRY(reg_setup(R, ctx, ref, rdims, rv, flo, fdims, fv, kFfdLevels, true, st));
  Mat A;
  memcpy(A.m, affine, sizeof(A.m));
  const double h0 = min_spacing(R.MR[0]);
  int lv[4];
  const int nl = used_levels(R, lv);
  float *grid = R.gbuf[0], *trial = R.gbuf[1], *dir = R.gbuf[2], *g = R.gbuf[3], *gn = R.gbuf[4];
  int32_t pg[3] = {0, 0, 0};
  for (int li = 0; li < nl; ++li) {
    const int l = lv[li];
    LevelInfo L;
    SC_TRY(level_info(R, l, L));
    int32_t gd[3];
    ffd_grid_dims(R.rd[l], gd);
    const int64_t ncp = (int64_t)gd[0] * gd[1] * gd[2], n = ncp * 3;
    if (li == 0) {
      SC_CUDA(cudaMemsetAsync(grid, 0, n * sizeof(float), st));
    } else {
      ProfScope ps(ctx, PC_REGISTER, st);
      subdivide_kernel<<<nblk(ncp, 128), 128, 0, st>>>(grid, pg[0], pg[1], pg[2], trial, gd[0], gd[1], gd[2]);
      ctx->launches++;
      SC_CUDA(cudaGetLastError());
      std::swap(grid, trial);
    }
    memcpy(pg, gd, sizeof(pg));
    auto value = [&](const float* gr, double& J) -> int {
      double nmi, be;
      SC_TRY(eval_be(R, gr, gd[0], gd[1], gd[2], be));
      SC_TRY(eval_nmi(R, make_geo(R, l, L, A, nullptr, gr), nmi));
      J = (1.0 - kLambda) * nmi - kLambda * be;
      return SC_OK;
    };
    auto grad = [&](const float* gr, float* out) -> int { return eval_grad(R, make_geo(R, l, L, A, nullptr, gr), nullptr, out); };
    const double h = h0 * (double)(1 << l);
    double J, alpha = kFfdAlpha0 * h, red[2];
    SC_TRY(value(grid, J));
    SC_TRY(grad(grid, g));
    SC_CUDA(cudaMemcpyAsync(dir, g, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    SC_TRY(vec_reduce(R, dir, nullptr, ncp, 1, red));
    double dn = red[0];
    int it = 0;
    while (it < kFfdIters && alpha >= kAlphaMin * h && dn > 0) {
      SC_TRY(axpy(R, trial, grid, alpha / dn, dir, n));
      double Jt;
      SC_TRY(value(trial, Jt));
      if (Jt > J) {
        std::swap(grid, trial);
        J = Jt; ++it;
        alpha = std::min(1.5 * alpha, kFfdAlphaMax * h);
        SC_TRY(grad(grid, gn));
        double gg[2], gx[2];
        SC_TRY(vec_reduce(R, g, g, ncp, 0, gg));     // g.g
        SC_TRY(vec_reduce(R, gn, g, ncp, 0, gx));    // gn.gn, gn.g
        const double beta = gg[0] > 0 ? std::max(0.0, (gx[0] - gx[1]) / gg[0]) : 0.0;
        SC_TRY(axpy(R, dir, gn, beta, dir, n));
        std::swap(g, gn);
        SC_TRY(vec_reduce(R, dir, nullptr, ncp, 1, red));
        dn = red[0];
      } else {
        alpha *= 0.5;
      }
    }
    ctx->reg_iters[4 + l] = it;
  }
  SC_CUDA(cudaMemcpyAsync(grid_out, grid, (size_t)pg[0] * pg[1] * pg[2] * 3 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return SC_OK;
}

int register_objective(sc_ctx* ctx, const float* ref, const int32_t* rdims, const double* rv, const float* flo, const int32_t* fdims,
                       const double* fv, const double* affine, const float* grid, double* value, double* agrad, float* ggrad,
                       cudaStream_t st) {
  Reg R;
  SC_TRY(reg_setup(R, ctx, ref, rdims, rv, flo, fdims, fv, 1, grid != nullptr, st));
  LevelInfo L;
  SC_TRY(level_info(R, 0, L));
  Mat A;
  memcpy(A.m, affine, sizeof(A.m));
  const Geo g = make_geo(R, 0, L, A, nullptr, grid);
  double nmi, be = 0.0;
  if (grid) SC_TRY(eval_be(R, grid, g.gx, g.gy, g.gz, be));
  SC_TRY(eval_nmi(R, g, nmi));
  value[0] = nmi; value[1] = be;
  value[2] = grid ? (1.0 - kLambda) * nmi - kLambda * be : nmi;
  if (agrad || ggrad) SC_TRY(eval_grad(R, g, agrad, ggrad));
  return SC_OK;
}

int warp_volume(sc_ctx* ctx, const float* flo, const int32_t* fdims, int C, const double* fv, const double* affine, const float* grid,
                const int32_t* rdims, const double* rv, float* out, cudaStream_t st) {
  Mat MR, MF, MFi, A;
  memcpy(MR.m, rv, sizeof(Mat)); memcpy(MF.m, fv, sizeof(Mat)); memcpy(A.m, affine, sizeof(Mat));
  SC_CHECK(inv4(MF, MFi), SC_ERR_ARG, "sc_warp_volume: flo_vox2mm is singular");
  Geo g{};
  g.rX = rdims[0]; g.rY = rdims[1]; g.rZ = rdims[2]; g.fX = fdims[0]; g.fY = fdims[1]; g.fZ = fdims[2];
  const Mat P = mul(MFi, mul(A, MR));
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 4; ++j) g.P[4 * i + j] = (float)P.m[4 * i + j];
    for (int j = 0; j < 3; ++j) g.Q[3 * i + j] = (float)MFi.m[4 * i + j];
  }
  int32_t gd[3];
  ffd_grid_dims(rdims, gd);
  g.grid = grid; g.gx = gd[0]; g.gy = gd[1]; g.gz = gd[2];
  ProfScope ps(ctx, PC_REGISTER, st);
  warp_kernel<<<nblk((int64_t)vox(rdims), 128), 128, 0, st>>>(g, flo, C, out);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

int prior_mask(sc_ctx* ctx, const float* priors, const int32_t* dims, int iterations, float* out, cudaStream_t st) {
  const int64_t n = (int64_t)vox(dims);
  SC_TRY(ensure_ws(ctx->ws_reg, 2 * ((n + 255) & ~(int64_t)255)));
  uint8_t* m = (uint8_t*)ctx->ws_reg.ptr;
  uint8_t* d = m + ((n + 255) & ~(int64_t)255);
  {
    ProfScope ps(ctx, PC_REGISTER, st);
    prior_any_kernel<<<nblk(n, 256), 256, 0, st>>>(priors, n, m);
    ctx->launches++;
  }
  SC_CUDA(cudaGetLastError());
  SC_TRY(launch_dilate(ctx, m, dims, iterations, d, st));
  {
    ProfScope ps(ctx, PC_REGISTER, st);
    u8_to_f32_kernel<<<nblk(n, 256), 256, 0, st>>>(d, n, out);
    ctx->launches++;
  }
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
