// K1: orthogonal patch gather + atlas vectors; candidate-voxel compaction; result scatter.
// Integer / byte work, HBM-write bound: no tensor cores here, only coalesced 128 B rows.
//
// Reference behaviour (paths relative to /root/reference):
//   get_patches        cnn_cort/base.py:272-308   window [c-16, c+16) on the two in-plane axes, zeros outside
//   atlas + bg-fix     cnn_cort/base.py:387-394   atlas[x,y,z,:]; if the row sums to 0 -> row[14] = 1
//   get_mask_voxels    cnn_cort/base.py:310-331   np.nonzero order (x slowest, z fastest)
//   scatter            cnn_cort/base.py:430-440
#include "common.cuh"

namespace sc {

constexpr int kGroup = 32;  // candidates per CTA

// One CTA (256 threads) gathers the three 32x32 views of kGroup candidates.  The kernel is bound by the patch
// WRITES (12 KB per candidate); everything is arranged so that a 128 B patch row costs a handful of instructions.
//  coronal  [dx][dz] at y and saggital [dy][dz] at x: a patch row is contiguous along z.  One warp copies one whole
//           patch (lane = column, loop over the 32 rows with running pointers): 128 B coalesced read (unaligned
//           start) -> 128 B streaming store per row.
//  axial    [dx][dy] at z: no contiguous in-plane axis.  Lanes run over the CANDIDATES instead (consecutive candidates
//           of np.nonzero order are consecutive in z => one 128 B line per load); every warp owns a private 32x33
//           shared tile that transposes one patch row index at a time, so the stores are again full patch rows and no
//           block-wide barrier is needed.
__global__ void __launch_bounds__(256) gather_patches_kernel(
    const float* __restrict__ vol, int X, int Y, int Z, const float* __restrict__ atlas, int bg_fix,
    const int32_t* __restrict__ xyz, int64_t n, float* __restrict__ ax, float* __restrict__ co,
    float* __restrict__ sa, float* __restrict__ atlas_out) {
  __shared__ int sx[kGroup], sy[kGroup], sz[kGroup];
  __shared__ float sbuf[8 * 32 * 33];                       // axial: 8 warp-private 32x33 tiles; fast path: the two 32x64 windows
  float (*tile)[32][33] = reinterpret_cast<float (*)[32][33]>(sbuf);
  __shared__ float satl[kGroup][16];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t ngroups = (n + kGroup - 1) / kGroup;
  // persistent CTAs: a grid of (resident CTAs per SM) x (SMs) walks the groups, no partial last wave
  for (int64_t grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
  const int64_t base = grp * kGroup;
  const int cnt = (int)min((int64_t)kGroup, n - base);
  __syncthreads();                                            // the previous group's shared data is no longer read
  if (tid < kGroup) {
    int64_t c = base + min(tid, cnt - 1);
    sx[tid] = xyz[c * 3 + 0];
    sy[tid] = xyz[c * 3 + 1];
    sz[tid] = xyz[c * 3 + 2];
  }
  __syncthreads();
  const int64_t YZ = (int64_t)Y * Z;

  // ---- coronal and saggital, fast path: a full group of candidates that are consecutive along z (the normal case in
  // np.nonzero order) shares 31/32 of its rows.  Stage the 32 x 63 window of each view once in shared memory and cut
  // the 32 patches out of it: the volume is read once per group instead of once per candidate (the kernel is bound by
  // the bytes moved through L2, reads included).
  float (*win)[32][64] = reinterpret_cast<float (*)[32][64]>(sbuf);
  const bool mine_ok = tid >= kGroup || (sx[tid] == sx[0] && sy[tid] == sy[0] && sz[tid] == sz[0] + tid);
  const bool run = __syncthreads_and(mine_ok && cnt == kGroup) != 0;
  if (run && (co || sa)) {
    const int x = sx[0], y = sy[0], z0 = sz[0];
    for (int e = tid; e < 2 * 32 * 64; e += 256) {
      const int view = e >> 11, i = (e >> 6) & 31, j = e & 63;
      const int zz = z0 - 16 + j;
      const int xx = view ? x : x - 16 + i, yy = view ? y - 16 + i : y;
      float v = 0.f;
      if (j < 63 && zz >= 0 && zz < Z && xx >= 0 && xx < X && yy >= 0 && yy < Y) v = __ldg(vol + (int64_t)xx * YZ + (int64_t)yy * Z + zz);
      win[view][i][j] = v;
    }
    __syncthreads();
    for (int job = warp; job < kGroup * 2; job += 8) {
      const int c = job >> 1, view = job & 1;
      float* dst = view ? sa : co;
      if (!dst) continue;
      float* out = dst + (base + c) * 1024 + lane;
      const float* src = &win[view][0][c + lane];
#pragma unroll 8
      for (int i = 0; i < 32; ++i) {
        __stcs(out, *src);
        src += 64;
        out += 32;
      }
    }
    __syncthreads();                                          // the axial tiles reuse the window's shared memory
  }

  // ---- coronal and saggital, general path: one warp per (candidate, view) ------------------------------
  for (int job = warp; job < (run ? 0 : cnt * 2); job += 8) {
    const int c = job >> 1, view = job & 1;
    float* dst = view ? sa : co;
    if (!dst) continue;
    const int x = sx[c], y = sy[c], z = sz[c];
    const int zz = z - 16 + lane;
    const bool zin = (zz >= 0) && (zz < Z);
    // view 0 (coronal): rows run over x at fixed y; view 1 (saggital): rows run over y at fixed x
    const int r0 = (view ? y : x) - 16, rmax = view ? Y : X;
    const int64_t rstride = view ? (int64_t)Z : YZ;
    const float* src = vol + (view ? (int64_t)x * YZ : (int64_t)y * Z) + (int64_t)r0 * rstride + zz;
    float* out = dst + (base + c) * 1024 + lane;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const int rr = r0 + i;
      float v = 0.f;
      if (zin && rr >= 0 && rr < rmax) v = __ldg(src);
      __stcs(out, v);
      src += rstride;
      out += 32;
    }
  }

  // ---- axial: lanes over candidates, transposed through a warp-private shared tile -------
  if (ax) {
    const int x = sx[lane], y = sy[lane], z = sz[lane];
    float (*tw)[33] = tile[warp];
    for (int i = warp; i < 32; i += 8) {
      const int xx = x - 16 + i;
      const bool xin = (xx >= 0) && (xx < X) && (lane < cnt);
      const float* src = vol + (int64_t)xx * YZ + (int64_t)(y - 16) * Z + z;
#pragma unroll 8
      for (int j = 0; j < 32; ++j) {
        const int yy = y - 16 + j;
        float v = 0.f;
        if (xin && yy >= 0 && yy < Y) v = __ldg(src);
        tw[j][lane] = v;
        src += Z;
      }
      __syncwarp();
      float* out = ax + base * 1024 + i * 32 + lane;
#pragma unroll 8
      for (int c = 0; c < 32; ++c) {
        if (c < cnt) __stcs(out, tw[lane][c]);
        out += 1024;
      }
      __syncwarp();
    }
  }

  // ---- atlas prior vector (+ background fix) ---------------------------------------------
  if (atlas_out) {
    for (int e = tid; e < cnt * 15; e += 256) {
      const int c = e / 15, ch = e - c * 15;
      const int64_t v = (int64_t)sx[c] * YZ + (int64_t)sy[c] * Z + sz[c];
      satl[c][ch] = __ldg(atlas + v * 15 + ch);
    }
    __syncthreads();
    if (bg_fix && tid < cnt) {
      // np.sum of a contiguous float32[15]: numpy's pairwise kernel keeps 8 partial sums for the
      // first 8 elements, combines them as a tree, then adds the remaining 7 in order.
      const float* a = satl[tid];
      float s = __fadd_rn(__fadd_rn(__fadd_rn(a[0], a[1]), __fadd_rn(a[2], a[3])),
                          __fadd_rn(__fadd_rn(a[4], a[5]), __fadd_rn(a[6], a[7])));
#pragma unroll
      for (int k = 8; k < 15; ++k) s = __fadd_rn(s, a[k]);
      if (s == 0.f) satl[tid][14] = 1.f;
    }
    __syncthreads();
    for (int e = tid; e < cnt * 15; e += 256) atlas_out[base * 15 + e] = satl[e / 15][e % 15];
  }
  }
}

int launch_gather(sc_ctx* ctx, const float* vol, const int32_t* dims, const float* atlas, int bg_fix,
                  const int32_t* xyz, int64_t n, float* ax, float* co, float* sa, float* atlas_out,
                  cudaStream_t st) {
  if (n == 0) return SC_OK;
  SC_CHECK(!atlas_out || atlas, SC_ERR_ARG, "sc_gather_patches: atlas output requested without an atlas");
  int64_t blocks = (n + kGroup - 1) / kGroup;
  const int64_t cap = (int64_t)ctx->sm_count * ctx->gather_ctas_per_sm;           // persistent CTAs (0 = one CTA per group)
  if (cap > 0 && blocks > cap) blocks = cap;
  SC_CHECK(blocks < (1ll << 31), SC_ERR_ARG, "sc_gather_patches: too many candidates in one call");
  ProfScope prof(ctx, PC_GATHER, st);
  gather_patches_kernel<<<(unsigned)blocks, 256, 0, st>>>(vol, dims[0], dims[1], dims[2], atlas, bg_fix, xyz, n, ax,
                                                          co, sa, atlas_out);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

__global__ void center_labels_kernel(const uint8_t* __restrict__ lab, int X, int Y, int Z, const int32_t* __restrict__ xyz,
                                     int64_t n, uint8_t* __restrict__ y) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int cx = xyz[i * 3], cy = xyz[i * 3 + 1], cz = xyz[i * 3 + 2];
  // a centre outside the volume reads the zero padding get_patches would have produced (base.py:303)
  if ((unsigned)cx >= (unsigned)X || (unsigned)cy >= (unsigned)Y || (unsigned)cz >= (unsigned)Z) { y[i] = 0; return; }
  y[i] = lab[((int64_t)cx * Y + cy) * Z + cz];
}

int launch_center_labels(sc_ctx* ctx, const uint8_t* lab, const int32_t* dims, const int32_t* xyz, int64_t n,
                         uint8_t* y, cudaStream_t st) {
  if (n == 0) return SC_OK;
  center_labels_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(lab, dims[0], dims[1], dims[2], xyz, n, y);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---- training minibatch from device-resident scans (sc_gather_samples) ---------------------------------------------
// Rows of a shuffled training set come from random voxels of several volumes, so nothing is shared between neighbouring
// samples (the np.nonzero-order fast paths of gather_patches_kernel never apply).  One warp per (sample, view), lane =
// patch column j, a loop over the 32 patch rows i; every store is one full 128 B patch row.
//   coronal  [dx][dz] at y, saggital [dy][dz] at x: the lanes read 32 consecutive z -> one 128 B line per row.
//   axial    [dx][dy] at z: the lanes stride by Z (one 32 B sector per element, 32 KB of sector traffic per patch).
// The warp of view 0 also passes the atlas row (lanes 0..14) and the label (lane 15) through.
__global__ void __launch_bounds__(256) gather_samples_kernel(
    const sc_scan* __restrict__ scans, int n_scans, const int32_t* __restrict__ samples, const float* __restrict__ atlas_rows,
    const uint8_t* __restrict__ labels, const int64_t* __restrict__ idx, int64_t n, float* __restrict__ ax,
    float* __restrict__ co, float* __restrict__ sa, float* __restrict__ atlas_out, uint8_t* __restrict__ y_out) {
  const int lane = threadIdx.x & 31;
  const int64_t job = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (job >= n * 3) return;
  const int64_t s = job / 3;
  const int view = (int)(job - s * 3);
  const int64_t r = idx ? __ldg(idx + s) : s;
  if (view == 0) {
    if (atlas_out && lane < 15) atlas_out[s * 15 + lane] = __ldg(atlas_rows + r * 15 + lane);
    if (y_out && lane == 15) y_out[s] = __ldg(labels + r);
  }
  float* dst = view == 0 ? ax : view == 1 ? co : sa;
  if (!dst) return;
  const int4 row = __ldg(reinterpret_cast<const int4*>(samples) + r);     // scan, x, y, z
  // an invalid scan index reads as an empty volume: zeros, never an out-of-bounds access
  const bool scan_ok = (unsigned)row.x < (unsigned)n_scans;
  const float* vol = nullptr;
  int X = 0, Y = 0, Z = 0;
  if (scan_ok) {
    vol = scans[row.x].vol;
    X = scans[row.x].dims[0]; Y = scans[row.x].dims[1]; Z = scans[row.x].dims[2];
  }
  const int64_t YZ = (int64_t)Y * Z;
  // patch row i runs along axis (ci, di, si), column j along (cj, dj, sj); (cf, df, sf) is the fixed axis of the slice
  int ci, di, cj, dj, cf, df;
  int64_t si, sj, sf;
  if (view == 0)      { ci = row.y; di = X; si = YZ; cj = row.z; dj = Y; sj = Z; cf = row.w; df = Z; sf = 1; }
  else if (view == 1) { ci = row.y; di = X; si = YZ; cj = row.w; dj = Z; sj = 1; cf = row.z; df = Y; sf = Z; }
  else                { ci = row.z; di = Y; si = Z;  cj = row.w; dj = Z; sj = 1; cf = row.y; df = X; sf = YZ; }
  const int jj = cj - 16 + lane;
  const bool jin = jj >= 0 && jj < dj && (unsigned)cf < (unsigned)df;
  const int i0 = ci - 16, imax = di;
  const float* src = vol + (int64_t)cf * sf + (int64_t)jj * sj + (int64_t)i0 * si;
  float* out = dst + s * 1024 + lane;
#pragma unroll 8
  for (int i = 0; i < 32; ++i) {
    const int ii = i0 + i;
    float v = 0.f;
    if (jin && ii >= 0 && ii < imax) v = __ldg(src);
    __stcs(out, v);
    src += si;
    out += 32;
  }
}

int launch_gather_samples(sc_ctx* ctx, const sc_scan* scans, int n_scans, const int32_t* samples, const float* atlas_rows,
                          const uint8_t* labels, const int64_t* idx, int64_t n, float* ax, float* co, float* sa,
                          float* atlas_out, uint8_t* y_out, cudaStream_t st) {
  if (n == 0) return SC_OK;
  const int64_t blocks = (n * 3 + 7) / 8;
  SC_CHECK(blocks < (1ll << 31), SC_ERR_ARG, "sc_gather_samples: too many samples in one call");
  ProfScope prof(ctx, PC_GATHER, st);
  gather_samples_kernel<<<(unsigned)blocks, 256, 0, st>>>(scans, n_scans, samples, atlas_rows, labels, idx, n, ax, co, sa,
                                                          atlas_out, y_out);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---------------------------------------------------------------------------------------
// Ordered stream compaction: count per 4096-element block, scan the block counts, emit.
// ---------------------------------------------------------------------------------------
constexpr int kNzPerThread = 16;
constexpr int kNzBlock = 256 * kNzPerThread;

template <int EB>
__device__ __forceinline__ bool nz_at(const void* vol, int64_t i) {
  if (EB == 1) return reinterpret_cast<const uint8_t*>(vol)[i] != 0;
  // float32 / int32: any non-zero bit pattern except -0.0f (numpy: -0.0 is False)
  uint32_t u = reinterpret_cast<const uint32_t*>(vol)[i];
  return (u & 0x7fffffffu) != 0;
}

template <int EB>
__global__ void __launch_bounds__(256) nz_count_kernel(const void* __restrict__ vol, int64_t total,
                                                       int32_t* __restrict__ counts) {
  const int64_t start = (int64_t)blockIdx.x * kNzBlock + (int64_t)threadIdx.x * kNzPerThread;
  int c = 0;
#pragma unroll
  for (int k = 0; k < kNzPerThread; ++k)
    if (start + k < total && nz_at<EB>(vol, start + k)) ++c;
  __shared__ int wsum[8];
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < 8; ++w) s += wsum[w];
    counts[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(1024) nz_scan_kernel(const int32_t* __restrict__ counts, int nblocks,
                                                       int64_t* __restrict__ offsets, int64_t* __restrict__ total) {
  __shared__ int64_t wsum[32];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < nblocks; b0 += 1024) {
    const int i = b0 + threadIdx.x;
    int64_t v = i < nblocks ? counts[i] : 0, inc = v;
    for (int o = 1; o < 32; o <<= 1) {
      int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if ((threadIdx.x & 31) >= o) inc += t;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
      int64_t w = wsum[threadIdx.x], winc = w;
      for (int o = 1; o < 32; o <<= 1) {
        int64_t t = __shfl_up_sync(0xffffffffu, winc, o);
        if (threadIdx.x >= o) winc += t;
      }
      wsum[threadIdx.x] = winc - w;
    }
    __syncthreads();
    const int64_t excl = carry + wsum[threadIdx.x >> 5] + inc - v;
    if (i < nblocks) offsets[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

template <int EB>
__global__ void __launch_bounds__(256) nz_emit_kernel(const void* __restrict__ vol, int64_t total, int Y, int Z,
                                                      const int64_t* __restrict__ offsets, int32_t* __restrict__ xyz,
                                                      int64_t capacity) {
  const int64_t start = (int64_t)blockIdx.x * kNzBlock + (int64_t)threadIdx.x * kNzPerThread;
  uint32_t bits = 0;
#pragma unroll
  for (int k = 0; k < kNzPerThread; ++k)
    if (start + k < total && nz_at<EB>(vol, start + k)) bits |= 1u << k;
  const int c = __popc(bits);
  int inc = c;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if ((threadIdx.x & 31) >= o) inc += t;
  }
  __shared__ int wsum[8];
  if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
  __syncthreads();
  int wbase = 0;
  for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) wbase += wsum[w];
  int64_t o = offsets[blockIdx.x] + wbase + inc - c;
  const int64_t YZ = (int64_t)Y * Z;
  while (bits) {
    const int k = __ffs(bits) - 1;
    bits &= bits - 1;
    const int64_t v = start + k;
    if (o < capacity) {
      const int x = (int)(v / YZ);
      const int64_t r = v - (int64_t)x * YZ;
      xyz[o * 3 + 0] = x;
      xyz[o * 3 + 1] = (int)(r / Z);
      xyz[o * 3 + 2] = (int)(r % Z);
    }
    ++o;
  }
}

int launch_nonzero(sc_ctx* ctx, const void* vol, int elem_bytes, const int32_t* dims, int32_t* xyz, int64_t capacity,
                   int64_t* n_out_host, cudaStream_t st) {
  SC_CHECK(elem_bytes == 1 || elem_bytes == 4, SC_ERR_ARG, "sc_nonzero_coords: elem_bytes must be 1 or 4");
  const int64_t total = (int64_t)dims[0] * dims[1] * dims[2];
  if (total == 0) {
    if (n_out_host) *n_out_host = 0;
    return SC_OK;
  }
  const int nblocks = (int)((total + kNzBlock - 1) / kNzBlock);
  SC_TRY(ensure_ws(ctx->ws, (size_t)nblocks * 12 + 64));
  int32_t* counts = reinterpret_cast<int32_t*>(ctx->ws.ptr);
  int64_t* offsets = reinterpret_cast<int64_t*>(reinterpret_cast<char*>(ctx->ws.ptr) + (((size_t)nblocks * 4 + 15) & ~(size_t)15));
  if (elem_bytes == 1) nz_count_kernel<1><<<nblocks, 256, 0, st>>>(vol, total, counts);
  else nz_count_kernel<4><<<nblocks, 256, 0, st>>>(vol, total, counts);
  nz_scan_kernel<<<1, 1024, 0, st>>>(counts, nblocks, offsets, ctx->d_count);
  if (xyz && capacity > 0) {
    if (elem_bytes == 1) nz_emit_kernel<1><<<nblocks, 256, 0, st>>>(vol, total, dims[1], dims[2], offsets, xyz, capacity);
    else nz_emit_kernel<4><<<nblocks, 256, 0, st>>>(vol, total, dims[1], dims[2], offsets, xyz, capacity);
    ctx->launches++;
  }
  ctx->launches += 2;
  SC_CUDA(cudaGetLastError());
  if (n_out_host) {
    SC_CUDA(cudaMemcpyAsync(ctx->h_count, ctx->d_count, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    SC_CUDA(cudaStreamSynchronize(st));
    *n_out_host = *ctx->h_count;
  }
  return SC_OK;
}

// ---- candidate rows of the dense path, compacted per slab (same order as np.nonzero inside the slab) -----------------
constexpr int kCmpBlock = 2048;          // dense rows per block: 256 threads x 8

__device__ __forceinline__ bool slab_cand(const uint8_t* __restrict__ cand, const OutGeo& g, int64_t plane, int ix0, int64_t m) {
  const int ix = (int)(m / plane);
  const int rem = (int)(m - (int64_t)ix * plane);
  const int iy = rem / g.bz, iz = rem - iy * g.bz;
  return cand[((int64_t)(g.x0 + ix0 + ix) * g.Y + (g.y0 + iy)) * g.Z + (g.z0 + iz)] != 0;
}

// pass 1 (emit == 0): candidates per block -> bc;  pass 3 (emit == 1): positions from the scanned block offsets
__global__ void __launch_bounds__(256) slab_compact_kernel(const uint8_t* __restrict__ cand, OutGeo g, int bx, int nxs, int bps,
                                                           int32_t* __restrict__ bc, const int32_t* __restrict__ boff,
                                                           int32_t* __restrict__ rowmap, int32_t* __restrict__ rowvox, int emit) {
  const int slab = blockIdx.x / bps, blk = blockIdx.x - slab * bps;
  const int64_t plane = (int64_t)g.by * g.bz;
  const int ix0 = slab * nxs;
  const int nx = bx - ix0 < nxs ? bx - ix0 : nxs;
  const int64_t rows = (int64_t)nx * plane, slab_base = (int64_t)ix0 * plane;
  const int64_t start = (int64_t)blk * kCmpBlock + (int64_t)threadIdx.x * 8;
  uint32_t bits = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (start + k < rows && slab_cand(cand, g, plane, ix0, start + k)) bits |= 1u << k;
  const int c = __popc(bits);
  int inc = c;
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if ((threadIdx.x & 31) >= o) inc += t;
  }
  __shared__ int wsum[8];
  if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
  __syncthreads();
  int wbase = 0, total = 0;
  for (int w = 0; w < 8; ++w) { if (w < (int)(threadIdx.x >> 5)) wbase += wsum[w]; total += wsum[w]; }
  if (!emit) {
    if (threadIdx.x == 0) bc[blockIdx.x] = total;
    return;
  }
  int o = boff[blockIdx.x] + wbase + inc - c;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (start + k >= rows) break;
    const bool on = (bits >> k) & 1u;
    rowmap[slab_base + start + k] = on ? o : -1;
    if (on) { rowvox[slab_base + o] = (int32_t)(start + k); ++o; }
  }
}

// pass 2: exclusive scan of the block counts of one slab (one CTA per slab), candidates of the slab -> cnt
__global__ void __launch_bounds__(1024) slab_scan_kernel(const int32_t* __restrict__ bc, int bps, int32_t* __restrict__ boff,
                                                         int32_t* __restrict__ cnt) {
  __shared__ int wsum[32];
  __shared__ int carry;
  const int32_t* c = bc + (int64_t)blockIdx.x * bps;
  int32_t* o = boff + (int64_t)blockIdx.x * bps;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < bps; b0 += 1024) {
    const int i = b0 + threadIdx.x;
    const int v = i < bps ? c[i] : 0;
    int inc = v;
    for (int s = 1; s < 32; s <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, s);
      if ((threadIdx.x & 31) >= s) inc += t;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
      const int w = wsum[threadIdx.x];
      int winc = w;
      for (int s = 1; s < 32; s <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, winc, s);
        if (threadIdx.x >= s) winc += t;
      }
      wsum[threadIdx.x] = winc - w;
    }
    __syncthreads();
    const int excl = carry + wsum[threadIdx.x >> 5] + inc - v;
    if (i < bps) o[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) cnt[blockIdx.x] = carry;
}

int launch_slab_compact(sc_ctx* ctx, const uint8_t* cand, const OutGeo& box, int bx, int nx_per_slab, int32_t* rowmap, int32_t* rowvox,
                        int32_t* cnt, int32_t* scratch, cudaStream_t st) {
  const int64_t plane = (int64_t)box.by * box.bz;
  const int nslabs = (bx + nx_per_slab - 1) / nx_per_slab;
  const int bps = (int)(((int64_t)nx_per_slab * plane + kCmpBlock - 1) / kCmpBlock);
  int32_t* bc = scratch;
  int32_t* boff = scratch + (int64_t)nslabs * bps;
  slab_compact_kernel<<<(unsigned)(nslabs * bps), 256, 0, st>>>(cand, box, bx, nx_per_slab, bps, bc, nullptr, nullptr, nullptr, 0);
  slab_scan_kernel<<<nslabs, 1024, 0, st>>>(bc, bps, boff, cnt);
  slab_compact_kernel<<<(unsigned)(nslabs * bps), 256, 0, st>>>(cand, box, bx, nx_per_slab, bps, bc, boff, rowmap, rowvox, 1);
  ctx->launches += 3;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// one iteration of scipy.ndimage.binary_dilation with the default (6-connected cross) structuring element and
// border_value 0: out = in | any face neighbour.  Ten iterations = the reference's crop mask (base.py:369).
__global__ void dilate6_kernel(const uint8_t* __restrict__ in, int X, int Y, int Z, uint8_t* __restrict__ out) {
  const int64_t total = (int64_t)X * Y * Z;
  const int64_t YZ = (int64_t)Y * Z;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += (int64_t)gridDim.x * blockDim.x) {
    const int x = (int)(v / YZ);
    const int r = (int)(v - (int64_t)x * YZ);
    const int y = r / Z, z = r - y * Z;
    uint8_t m = in[v];
    if (!m) {
      m = (x > 0 && in[v - YZ]) || (x + 1 < X && in[v + YZ]) || (y > 0 && in[v - Z]) || (y + 1 < Y && in[v + Z]) ||
          (z > 0 && in[v - 1]) || (z + 1 < Z && in[v + 1]);
    }
    out[v] = m ? 1 : 0;
  }
}

int launch_dilate(sc_ctx* ctx, const uint8_t* mask, const int32_t* dims, int iterations, uint8_t* out, cudaStream_t st) {
  const int64_t total = (int64_t)dims[0] * dims[1] * dims[2];
  SC_CHECK(iterations >= 0, SC_ERR_ARG, "sc_dilate_mask: negative iteration count");
  if (iterations == 0) {
    SC_CUDA(cudaMemcpyAsync(out, mask, total, cudaMemcpyDeviceToDevice, st));
    return SC_OK;
  }
  SC_TRY(ensure_ws(ctx->ws, (size_t)total + 256));
  uint8_t* tmp = reinterpret_cast<uint8_t*>(ctx->ws.ptr);
  const unsigned grid = (unsigned)((total + 255) / 256 < (int64_t)ctx->sm_count * 32 ? (total + 255) / 256 : (int64_t)ctx->sm_count * 32);
  const uint8_t* src = mask;
  for (int i = 0; i < iterations; ++i) {   // ping-pong so that the last iteration lands in `out`
    uint8_t* dst = ((iterations - 1 - i) & 1) ? tmp : out;
    dilate6_kernel<<<grid, 256, 0, st>>>(src, dims[0], dims[1], dims[2], dst);
    ctx->launches++;
    src = dst;
  }
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

__global__ void scatter_kernel(const int32_t* __restrict__ xyz, int64_t n, const int32_t* __restrict__ label,
                               const float* __restrict__ proba, int X, int Y, int Z, uint8_t* __restrict__ label_vol,
                               float* __restrict__ proba_vol) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int cx = xyz[i * 3], cy = xyz[i * 3 + 1], cz = xyz[i * 3 + 2];
  if ((unsigned)cx >= (unsigned)X || (unsigned)cy >= (unsigned)Y || (unsigned)cz >= (unsigned)Z) return;   // numpy would raise; never write out of bounds
  const int64_t v = ((int64_t)cx * Y + cy) * Z + cz;
  if (label_vol && label) label_vol[v] = (uint8_t)label[i];
  if (proba_vol && proba) {
#pragma unroll
    for (int c = 0; c < 15; ++c) proba_vol[v * 15 + c] = proba[i * 15 + c];
  }
}

int launch_scatter(sc_ctx* ctx, const int32_t* xyz, int64_t n, const int32_t* label, const float* proba,
                   const int32_t* dims, uint8_t* label_vol, float* proba_vol, cudaStream_t st) {
  if (n == 0) return SC_OK;
  ProfScope prof(ctx, PC_SCATTER, st);
  scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(xyz, n, label, proba, dims[0], dims[1], dims[2], label_vol,
                                                              proba_vol);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
