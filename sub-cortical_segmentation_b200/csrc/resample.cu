// Resampling between a scan's native grid and the isotropic grid the network runs on (DESIGN.md section 13).
//
// Per axis a native extent n maps to m target voxels, r = n / m; both grids cover the same field of view.
//   native -> target: target j sits at native x_j = (j + 0.5) r - 0.5; out_j = sum_i w_ij v_i / sum_i w_ij with
//     w_ij = max(0, 1 - |i - x_j| / h), h = max(r, 1): an antialiasing triangle filter when shrinking, linear interpolation
//     with the edge value held when growing, the identity when r = 1.  Separable: one pass per axis.
//   target -> native: native v sits at target y = clamp((v + 0.5) / r - 0.5, 0, m - 1); the probability vector is the
//     trilinear mean over the neighbours with non-zero weight that are target candidates, renormalised; label = first arg-max.
// The host builds the per-axis tables in double and uploads them as int32 / float32; the kernels accumulate in fp32 in a
// fixed order without atomics, so the same inputs give byte-identical outputs.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace sc {

// one pass along the middle axis of a volume viewed as [outer][n][inner] (inner = the faster axes times the channels) ->
// [outer][m][inner]: one thread per output element, inner index fastest (coalesced loads and stores)
__global__ void __launch_bounds__(256) resample_axis_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t total,
                                                            int64_t inner, int n, int m, const int32_t* __restrict__ first,
                                                            const int32_t* __restrict__ count, const float* __restrict__ w, int K) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= total) return;
  const int64_t q = o % inner, t = o / inner;
  const int j = (int)(t % m);
  const int64_t outer = t / m;
  const float* src = in + (outer * n + first[j]) * inner + q;
  const float* wj = w + (int64_t)j * K;
  const int c = count[j];
  float acc = 0.f;
  for (int k = 0; k < c; ++k) acc = fmaf(wj[k], __ldg(src + (int64_t)k * inner), acc);
  out[o] = acc;
}

// one thread per native voxel, z fastest; tables: i0[nX + nY + nZ] (lower target neighbour) and f[...] (weight of the upper one)
__global__ void __launch_bounds__(256) map_back_kernel(const float* __restrict__ proba, const uint8_t* __restrict__ cand, int tY, int tZ,
                                                       const uint8_t* __restrict__ nmask, int nX, int nY, int nZ,
                                                       const int32_t* __restrict__ i0, const float* __restrict__ f,
                                                       uint8_t* __restrict__ label, float* __restrict__ pout) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= (int64_t)nX * nY * nZ) return;
  if (nmask && !nmask[v]) return;
  const int z = (int)(v % nZ), y = (int)((v / nZ) % nY), x = (int)(v / ((int64_t)nY * nZ));
  const int ix = i0[x], iy = i0[nX + y], iz = i0[nX + nY + z];
  const float fx = f[x], fy = f[nX + y], fz = f[nX + nY + z];
  float acc[15];
#pragma unroll
  for (int c = 0; c < 15; ++c) acc[c] = 0.f;
  float wsum = 0.f;
#pragma unroll
  for (int d = 0; d < 8; ++d) {
    const int dx = d >> 2, dy = (d >> 1) & 1, dz = d & 1;
    const float wt = (dx ? fx : 1.f - fx) * (dy ? fy : 1.f - fy) * (dz ? fz : 1.f - fz);
    if (wt <= 0.f) continue;                 // a zero-weight corner is no neighbour (and may lie outside the grid)
    const int64_t t = ((int64_t)(ix + dx) * tY + (iy + dy)) * tZ + (iz + dz);
    if (!cand[t]) continue;
    wsum += wt;
    const float* p = proba + t * 15;
#pragma unroll
    for (int c = 0; c < 15; ++c) acc[c] = fmaf(wt, __ldg(p + c), acc[c]);
  }
  if (wsum <= 0.f) return;
  const float inv = 1.f / wsum;
  int best = 0;
  float bp = acc[0] * inv;
#pragma unroll
  for (int c = 0; c < 15; ++c) {
    acc[c] *= inv;
    if (acc[c] > bp) { bp = acc[c]; best = c; }
  }
  label[v] = (uint8_t)best;
  if (pout) {
#pragma unroll
    for (int c = 0; c < 15; ++c) pout[v * 15 + c] = acc[c];
  }
}

namespace {

// tap table of one native -> target axis (n -> m): first tap, tap count and normalised weights, K taps per row (zero padded)
struct Taps { std::vector<int32_t> first, count; std::vector<float> w; int K = 0; };

Taps make_taps(int n, int m) {
  Taps T;
  const double r = (double)n / m, h = std::max(r, 1.0);
  std::vector<std::vector<double>> rows(m);
  T.first.resize(m);
  T.count.resize(m);
  for (int j = 0; j < m; ++j) {
    const double x = (j + 0.5) * r - 0.5;
    int lo = std::max(0, (int)floor(x - h)), hi = std::min(n - 1, (int)ceil(x + h));
    while (lo < hi && 1.0 - fabs(lo - x) / h <= 0.0) ++lo;
    while (hi > lo && 1.0 - fabs(hi - x) / h <= 0.0) --hi;
    double s = 0.0;
    for (int i = lo; i <= hi; ++i) { rows[j].push_back(std::max(0.0, 1.0 - fabs(i - x) / h)); s += rows[j].back(); }
    for (double& v : rows[j]) v /= s;
    T.first[j] = lo;
    T.count[j] = hi - lo + 1;
    T.K = std::max(T.K, T.count[j]);
  }
  T.w.assign((size_t)m * T.K, 0.f);
  for (int j = 0; j < m; ++j)
    for (int k = 0; k < T.count[j]; ++k) T.w[(size_t)j * T.K + k] = (float)rows[j][k];
  return T;
}

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

int resample_volume(sc_ctx* ctx, const float* in, const int32_t* in_dims, int channels, const int32_t* out_dims, float* out,
                    cudaStream_t st) {
  int order[3], np = 0;
  for (int a = 0; a < 3; ++a)
    if (in_dims[a] != out_dims[a]) order[np++] = a;
  const int64_t nin = (int64_t)in_dims[0] * in_dims[1] * in_dims[2] * channels;
  if (np == 0) {                              // every axis has r = 1: the identity
    SC_CUDA(cudaMemcpyAsync(out, in, (size_t)nin * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return SC_OK;
  }
  // the axes that shrink most go first: every later pass then reads and writes the fewest elements
  std::sort(order, order + np, [&](int a, int b) {
    return std::make_pair((double)out_dims[a] / in_dims[a], a) < std::make_pair((double)out_dims[b] / in_dims[b], b);
  });
  // tables of all passes in one upload, then two ping-pong intermediates
  Taps T[3];
  size_t tab_off[3], tab_bytes = 0;
  for (int p = 0; p < np; ++p) {
    const int a = order[p];
    T[p] = make_taps(in_dims[a], out_dims[a]);
    tab_off[p] = tab_bytes;
    tab_bytes += align256((size_t)out_dims[a] * 8 + T[p].w.size() * sizeof(float));
  }
  int32_t cur[3] = {in_dims[0], in_dims[1], in_dims[2]};
  int64_t inter = 0;
  for (int p = 0; p + 1 < np; ++p) {
    cur[order[p]] = out_dims[order[p]];
    inter = std::max(inter, (int64_t)cur[0] * cur[1] * cur[2] * channels);
  }
  const size_t ib = align256((size_t)inter * sizeof(float));
  SC_TRY(ensure_ws(ctx->ws_resample, tab_bytes + 2 * ib));
  char* base = static_cast<char*>(ctx->ws_resample.ptr);
  std::vector<char> host(tab_bytes, 0);
  for (int p = 0; p < np; ++p) {
    const int m = out_dims[order[p]];
    char* h = host.data() + tab_off[p];
    memcpy(h, T[p].first.data(), (size_t)m * 4);
    memcpy(h + (size_t)m * 4, T[p].count.data(), (size_t)m * 4);
    memcpy(h + (size_t)m * 8, T[p].w.data(), T[p].w.size() * sizeof(float));
  }
  SC_CUDA(cudaMemcpyAsync(base, host.data(), tab_bytes, cudaMemcpyHostToDevice, st));
  float* buf[2] = {reinterpret_cast<float*>(base + tab_bytes), reinterpret_cast<float*>(base + tab_bytes + ib)};
  int32_t d[3] = {in_dims[0], in_dims[1], in_dims[2]};
  const float* src = in;
  for (int p = 0; p < np; ++p) {
    const int a = order[p], n = d[a], m = out_dims[a];
    int64_t inner = channels;
    for (int b = a + 1; b < 3; ++b) inner *= d[b];
    d[a] = m;
    const int64_t total = (int64_t)d[0] * d[1] * d[2] * channels;
    float* dst = p + 1 == np ? out : buf[p & 1];
    const char* tb = base + tab_off[p];
    ProfScope prof(ctx, PC_RESAMPLE, st);
    resample_axis_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
        src, dst, total, inner, n, m, reinterpret_cast<const int32_t*>(tb), reinterpret_cast<const int32_t*>(tb + (size_t)m * 4),
        reinterpret_cast<const float*>(tb + (size_t)m * 8), T[p].K);
    SC_CUDA(cudaGetLastError());
    ctx->launches++;
    src = dst;
  }
  return SC_OK;
}

int map_proba_back(sc_ctx* ctx, const float* proba, const uint8_t* cand, const int32_t* tdims, const uint8_t* nmask,
                   const int32_t* ndims, uint8_t* label, float* pout, cudaStream_t st) {
  const int ntot = ndims[0] + ndims[1] + ndims[2];
  std::vector<int32_t> i0(ntot);
  std::vector<float> f(ntot);
  for (int a = 0, o = 0; a < 3; o += ndims[a], ++a) {
    const int n = ndims[a], m = tdims[a];
    const double r = (double)n / m;
    for (int v = 0; v < n; ++v) {
      const double y = std::min(std::max((v + 0.5) / r - 0.5, 0.0), (double)(m - 1));
      const int lo = m > 1 ? std::min((int)floor(y), m - 2) : 0;
      i0[o + v] = lo;
      f[o + v] = (float)(y - lo);
    }
  }
  const size_t fo = align256((size_t)ntot * 4);
  SC_TRY(ensure_ws(ctx->ws_resample, fo + (size_t)ntot * 4));
  char* base = static_cast<char*>(ctx->ws_resample.ptr);
  std::vector<char> host(fo + (size_t)ntot * 4, 0);
  memcpy(host.data(), i0.data(), (size_t)ntot * 4);
  memcpy(host.data() + fo, f.data(), (size_t)ntot * 4);
  SC_CUDA(cudaMemcpyAsync(base, host.data(), host.size(), cudaMemcpyHostToDevice, st));
  const int64_t nv = (int64_t)ndims[0] * ndims[1] * ndims[2];
  ProfScope prof(ctx, PC_RESAMPLE, st);
  map_back_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(proba, cand, tdims[1], tdims[2], nmask, ndims[0], ndims[1], ndims[2],
                                                                 reinterpret_cast<const int32_t*>(base), reinterpret_cast<const float*>(base + fo),
                                                                 label, pout);
  SC_CUDA(cudaGetLastError());
  ctx->launches++;
  return SC_OK;
}

}  // namespace sc
