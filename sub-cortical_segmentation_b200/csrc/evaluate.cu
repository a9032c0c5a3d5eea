// Segmentation metrics on the device (sc_evaluate_segmentation): per structure l = 1..14 of two label volumes seg / ref
// (15 counts as 0), voxel counts, Dice, volumes and the surface distances d_AB / d_BA between S(A) = surface of
// (seg == l) and S(B) = surface of (ref == l), with hd, hd95 (numpy's linear percentile) and assd.  The definitions are
// those of oracle/evaluate.py (scipy binary_erosion + distance_transform_edt), checked number for number.
//
//   1. eval_surface_kernel: one pass over both volumes -> 15x15 confusion counts, labels > 15, the surface byte map
//      (bit 0: seg's class has a surface voxel here, bit 1: ref's class), per class the surface counts and the bounding
//      box of S(A) | S(B).  One host synchronise reads these.
//   2. per class with A and B non-empty, on that box and for both directions at once (blockIdx.y): an exact separable
//      Euclidean distance transform of the feature surface in float64 with the spacing weights -- nearest feature along x,
//      then a lower envelope of parabolas (Felzenszwalb-Huttenlocher) along y and along z; one thread per line, adjacent
//      threads on adjacent lines, the envelope stacks in the workspace as [k][line].  The z pass samples the query
//      surface directly: count, sum and max per direction, and every distance appended to the class's list.
//   3. hd95: radix select (8-bit digits over the IEEE bits of the non-negative doubles, shared-memory histograms) of the
//      order statistic at floor(h) and a min-reduction for the one after it; numpy's interpolation on the host.
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace sc {

constexpr int kFar = 0x7fffffff;          // no feature on the x line
constexpr int kEdtThreads = 128;

struct EvalCounts {                        // phase 1, zeroed per call
  unsigned long long conf[225];            // [ref class][seg class], 15 -> 0
  unsigned long long invalid[2];           // voxels with a label > 15 in seg / ref
  unsigned long long nsurf[2][16];         // surface voxels of each class in seg / ref
  int box[16][6];                          // per class: half-open box {x0,x1,y0,y1,z0,z1} of S(A) | S(B)
};
struct EvalDist {                          // phases 2 and 3, zeroed per call
  unsigned long long cnt[16][2];           // per class and direction (0: d_AB, 1: d_BA)
  double sum[16][2];
  unsigned long long max[16][2];           // bits of a non-negative double: they order as the values do
  unsigned long long list_n[16];           // distances appended to the class's list
  unsigned long long prefix[16];           // radix select: key bits fixed so far; after the last digit the selected key
  unsigned long long rank[16];             // rank still to find among the keys that share the prefix
  unsigned long long list_off[16];         // start of the class's list (set with rank by the host)
  unsigned long long le[16];               // keys <= the selected key
  unsigned long long gt_min[16];           // smallest key above it
  unsigned long long hist[16][256];
};
struct EvalBox { int x0, y0, z0, bx, by, bz; };

__global__ void eval_init_kernel(EvalCounts* __restrict__ c, EvalDist* __restrict__ d, int X, int Y, int Z) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(c);
  for (int i = threadIdx.x; i < (int)(offsetof(EvalCounts, box) / 8); i += blockDim.x) a[i] = 0;
  for (int i = threadIdx.x; i < 16 * 6; i += blockDim.x) {
    const int k = i % 6, dim = k < 2 ? X : k < 4 ? Y : Z;
    c->box[i / 6][k] = (k & 1) ? 0 : dim;
  }
  unsigned long long* b = reinterpret_cast<unsigned long long*>(d);
  for (int i = threadIdx.x; i < (int)(sizeof(EvalDist) / 8); i += blockDim.x) b[i] = 0;
  __syncthreads();
  if (threadIdx.x < 16) d->gt_min[threadIdx.x] = ~0ull;
}

// v is on the surface of its class c (1..14) in `lab`: a 6-neighbour outside the volume or with another label
// (a neighbour holding 15 has class 0 != c)
__device__ __forceinline__ bool on_surface(const uint8_t* __restrict__ lab, int64_t v, int x, int y, int z, int X, int Y, int Z,
                                           int64_t YZ, int c) {
  if (x == 0 || y == 0 || z == 0 || x == X - 1 || y == Y - 1 || z == Z - 1) return true;
  return lab[v - 1] != c || lab[v + 1] != c || lab[v - Z] != c || lab[v + Z] != c || lab[v - YZ] != c || lab[v + YZ] != c;
}

__device__ __forceinline__ void box_add(int* b, int x, int y, int z) {
  atomicMin(&b[0], x); atomicMax(&b[1], x + 1);
  atomicMin(&b[2], y); atomicMax(&b[3], y + 1);
  atomicMin(&b[4], z); atomicMax(&b[5], z + 1);
}

// phase 1.  The loop bound is uniform per block, so every lane of a warp takes part in the __match_any_sync that
// aggregates the confusion increments (most voxels of a warp share one bin)
__global__ void __launch_bounds__(256) eval_surface_kernel(const uint8_t* __restrict__ seg, const uint8_t* __restrict__ ref, int X, int Y,
                                                           int Z, uint8_t* __restrict__ surf, EvalCounts* __restrict__ out) {
  __shared__ unsigned s_conf[225];
  __shared__ unsigned s_inv[2];
  __shared__ unsigned s_ns[2][16];
  __shared__ int s_box[16][6];
  for (int i = threadIdx.x; i < 225; i += blockDim.x) s_conf[i] = 0;
  if (threadIdx.x < 2) s_inv[threadIdx.x] = 0;
  if (threadIdx.x < 32) s_ns[threadIdx.x >> 4][threadIdx.x & 15] = 0;
  if (threadIdx.x < 96) {
    const int k = threadIdx.x % 6;
    s_box[threadIdx.x / 6][k] = (k & 1) ? 0 : (k < 2 ? X : k < 4 ? Y : Z);
  }
  __syncthreads();
  const int64_t YZ = (int64_t)Y * Z, total = (int64_t)X * YZ;
  const int lane = threadIdx.x & 31;
  for (int64_t v0 = (int64_t)blockIdx.x * blockDim.x; v0 < total; v0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = v0 + threadIdx.x;
    int key = -1;
    if (v < total) {
      const int x = (int)(v / YZ), r = (int)(v - x * YZ), y = r / Z, z = r - y * Z;
      const int s = seg[v], t = ref[v];
      if (s > 15) atomicAdd(&s_inv[0], 1u);
      if (t > 15) atomicAdd(&s_inv[1], 1u);
      const int sc = s == 15 ? 0 : s, tc = t == 15 ? 0 : t;
      if (s <= 15 && t <= 15) key = tc * 15 + sc;
      uint8_t bits = 0;
      if (sc >= 1 && sc <= 14 && on_surface(seg, v, x, y, z, X, Y, Z, YZ, sc)) {
        bits |= 1;
        atomicAdd(&s_ns[0][sc], 1u);
        box_add(s_box[sc], x, y, z);
      }
      if (tc >= 1 && tc <= 14 && on_surface(ref, v, x, y, z, X, Y, Z, YZ, tc)) {
        bits |= 2;
        atomicAdd(&s_ns[1][tc], 1u);
        box_add(s_box[tc], x, y, z);
      }
      surf[v] = bits;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && lane == __ffs(peers) - 1) atomicAdd(&s_conf[key], (unsigned)__popc(peers));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 225; i += blockDim.x)
    if (s_conf[i]) atomicAdd(&out->conf[i], (unsigned long long)s_conf[i]);
  if (threadIdx.x < 2 && s_inv[threadIdx.x]) atomicAdd(&out->invalid[threadIdx.x], (unsigned long long)s_inv[threadIdx.x]);
  if (threadIdx.x < 32) {
    const int w = threadIdx.x >> 4, c = threadIdx.x & 15;
    if (s_ns[w][c]) atomicAdd(&out->nsurf[w][c], (unsigned long long)s_ns[w][c]);
  }
  if (threadIdx.x < 16 && s_box[threadIdx.x][1] > 0) {
    int* b = out->box[threadIdx.x];
    const int* sb = s_box[threadIdx.x];
    atomicMin(&b[0], sb[0]); atomicMax(&b[1], sb[1]);
    atomicMin(&b[2], sb[2]); atomicMax(&b[3], sb[3]);
    atomicMin(&b[4], sb[4]); atomicMax(&b[5], sb[5]);
  }
}

// phase 2a: distance in voxels to the nearest feature on each x line of the box (kFar: none).  Lines (iy, iz), field
// g[dir][ix][iy][iz].  Features of direction 0 (d_AB) are S(B): ref == cls with bit 1; of direction 1 S(A)
__global__ void __launch_bounds__(kEdtThreads) edt_x_kernel(const uint8_t* __restrict__ seg, const uint8_t* __restrict__ ref,
                                                            const uint8_t* __restrict__ surf, int Y, int Z, EvalBox b, int cls,
                                                            int* __restrict__ g) {
  const int64_t nl = (int64_t)b.by * b.bz;
  const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= nl) return;
  const int dir = blockIdx.y, bit = dir == 0 ? 2 : 1;
  const uint8_t* __restrict__ lab = dir == 0 ? ref : seg;
  const int iy = (int)(line / b.bz), iz = (int)(line - (int64_t)iy * b.bz);
  const int64_t YZ = (int64_t)Y * Z;
  const int64_t v0 = ((int64_t)b.x0 * Y + b.y0 + iy) * Z + b.z0 + iz;
  int* __restrict__ o = g + (int64_t)dir * b.bx * nl + line;
  int last = -1;
  for (int ix = 0; ix < b.bx; ++ix) {
    const int64_t v = v0 + ix * YZ;
    if ((surf[v] & bit) && lab[v] == cls) last = ix;
    o[ix * nl] = last < 0 ? kFar : ix - last;
  }
  int next = -1;
  for (int ix = b.bx - 1; ix >= 0; --ix) {
    const int d = o[ix * nl];
    if (d == 0) next = ix;
    else if (next >= 0 && next - ix < d) o[ix * nl] = next - ix;
  }
}

// Lower envelope of the parabolas w^2 (q - i)^2 + f_i over the finite f_i of one line (element i at f[i * stride]); the stack
// of line `line` is entry k at [k * nl + line] of sv / sf / sz (vertex, its f, left boundary in index units).  -> entries - 1
__device__ __forceinline__ int envelope_build(const double* __restrict__ f, int64_t stride, int n, double w2, int64_t nl, int64_t line,
                                              int* __restrict__ sv, double* __restrict__ sf, double* __restrict__ sz) {
  int k = -1, vk = 0;
  double fk = 0.0, zk = 0.0;
  for (int q = 0; q < n; ++q) {
    const double fq = f[q * stride];
    if (isinf(fq)) continue;
    double s = 0.0;
    while (k >= 0) {
      s = ((fq + w2 * q * q) - (fk + w2 * vk * vk)) / (2.0 * w2 * (q - vk));
      if (k == 0 || s > zk) break;
      --k;                                               // the top parabola is hidden: pop it
      vk = sv[k * nl + line]; fk = sf[k * nl + line]; zk = sz[k * nl + line];
    }
    ++k;
    vk = q; fk = fq; zk = s;
    sv[k * nl + line] = q; sf[k * nl + line] = fq; sz[k * nl + line] = s;
  }
  return k;
}

// walks the envelope in order of increasing q: the parabola j in force at q and its squared distance, rounded as
// scipy rounds sum((delta * w)^2) (no fused multiply-add)
struct EnvelopeCursor {
  const int* sv; const double* sf; const double* sz; int64_t nl, line; int top, j, vj; double fj, znext, w;
  __device__ void init(int k) {
    top = k; j = 0;
    vj = sv[line]; fj = sf[line];
    znext = top > 0 ? sz[nl + line] : INFINITY;
  }
  __device__ double at(int q) {
    while (znext < q) {
      ++j;
      vj = sv[j * nl + line]; fj = sf[j * nl + line];
      znext = j < top ? sz[(j + 1) * nl + line] : INFINITY;
    }
    const double dd = __dmul_rn(w, (double)(q - vj));
    return __dadd_rn(__dmul_rn(dd, dd), fj);
  }
};

// phase 2b: lines (ix, iz) along y; h[dir][ix][iy][iz] = min over the x line distances of g, squared in mm^2
__global__ void __launch_bounds__(kEdtThreads) edt_y_kernel(const int* __restrict__ g, EvalBox b, double sx, double sy,
                                                            double* __restrict__ h, int* __restrict__ sv, double* __restrict__ sf,
                                                            double* __restrict__ sz) {
  const int64_t nl = (int64_t)b.bx * b.bz;
  const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= nl) return;
  const int dir = blockIdx.y;
  const int ix = (int)(line / b.bz), iz = (int)(line - (int64_t)ix * b.bz);
  const int64_t vol = (int64_t)b.bx * b.by * b.bz;
  const int64_t base = (int64_t)dir * vol + (int64_t)ix * b.by * b.bz + iz;
  const int* __restrict__ gi = g + base;
  double* __restrict__ ho = h + base;
  // the x distances become f values: written into h first (the envelope reads them from there), overwritten below
  for (int iy = 0; iy < b.by; ++iy) {
    const int d = gi[(int64_t)iy * b.bz];
    const double dx = __dmul_rn(sx, (double)d);
    ho[(int64_t)iy * b.bz] = d == kFar ? INFINITY : __dmul_rn(dx, dx);
  }
  const int64_t so = (int64_t)dir * b.by * nl;
  const int k = envelope_build(ho, b.bz, b.by, sy * sy, nl, line, sv + so, sf + so, sz + so);
  if (k < 0) return;                                      // no feature in this (x, y) plane column: h stays infinite
  EnvelopeCursor e{sv + so, sf + so, sz + so, nl, line, 0, 0, 0, 0.0, 0.0, sy};
  e.init(k);
  for (int iy = 0; iy < b.by; ++iy) ho[(int64_t)iy * b.bz] = e.at(iy);
}

// phase 2c: lines (ix, iy) along z; samples the query surface (direction 0: S(A) = seg == cls with bit 0) and appends each
// distance to the class's list.  Every lane of a warp walks the same z range so that the appends aggregate per warp.
__global__ void __launch_bounds__(kEdtThreads) edt_z_kernel(const uint8_t* __restrict__ seg, const uint8_t* __restrict__ ref,
                                                            const uint8_t* __restrict__ surf, int Y, int Z, EvalBox b, int cls, double sz_w,
                                                            const double* __restrict__ h, int* __restrict__ sv, double* __restrict__ sf,
                                                            double* __restrict__ szb, double* __restrict__ list, EvalDist* __restrict__ dist) {
  const int64_t nl = (int64_t)b.bx * b.by;
  const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = line < nl;
  const int dir = blockIdx.y, bit = dir == 0 ? 1 : 2;
  const uint8_t* __restrict__ lab = dir == 0 ? seg : ref;
  const int64_t vol = (int64_t)b.bx * b.by * b.bz;
  const int64_t so = (int64_t)dir * b.bz * nl;
  int k = -1;
  int64_t v0 = 0;
  EnvelopeCursor e{sv + so, sf + so, szb + so, nl, line, 0, 0, 0, 0.0, 0.0, sz_w};
  if (live) {
    const int ix = (int)(line / b.by), iy = (int)(line - (int64_t)ix * b.by);
    k = envelope_build(h + (int64_t)dir * vol + line * b.bz, 1, b.bz, sz_w * sz_w, nl, line, sv + so, sf + so, szb + so);
    if (k >= 0) e.init(k);
    v0 = ((int64_t)(b.x0 + ix) * Y + b.y0 + iy) * Z + b.z0;
  }
  const int lane = threadIdx.x & 31;
  unsigned long long cnt = 0;
  double sum = 0.0, mx = 0.0;
  for (int iz = 0; iz < b.bz; ++iz) {
    bool q = false;
    double d = 0.0;
    if (k >= 0) {
      const int64_t v = v0 + iz;
      if ((surf[v] & bit) && lab[v] == cls) {
        d = sqrt(e.at(iz));
        q = true;
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, q);
    if (m) {
      const int leader = __ffs(m) - 1;
      unsigned long long at = 0;
      if (lane == leader) at = atomicAdd(&dist->list_n[cls], (unsigned long long)__popc(m));
      at = __shfl_sync(0xffffffffu, at, leader);
      if (q) {
        list[at + __popc(m & ((1u << lane) - 1u))] = d;
        ++cnt; sum += d; mx = fmax(mx, d);
      }
    }
  }
  for (int o = 16; o; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if (lane == 0 && cnt) {
    atomicAdd(&dist->cnt[cls][dir], cnt);
    atomicAdd(&dist->sum[cls][dir], sum);
    atomicMax(&dist->max[cls][dir], (unsigned long long)__double_as_longlong(mx));
  }
}

// phase 3: one 8-bit digit of the radix select, all classes at once (blockIdx.y = class - 1).  Keys whose higher digits
// equal the prefix are counted by their digit at `shift`.
__global__ void __launch_bounds__(256) select_hist_kernel(const double* __restrict__ list, EvalDist* __restrict__ dist, int shift) {
  __shared__ unsigned hs[256];
  const int c = blockIdx.y + 1;
  const unsigned long long n = dist->list_n[c];
  if (n == 0) return;                                     // uniform per block
  hs[threadIdx.x] = 0;
  __syncthreads();
  const unsigned long long pre = dist->prefix[c], hi = shift == 56 ? 0ull : ~0ull << (shift + 8);
  const unsigned long long* __restrict__ keys = reinterpret_cast<const unsigned long long*>(list + dist->list_off[c]);
  const int lane = threadIdx.x & 31;
  for (unsigned long long i0 = (unsigned long long)blockIdx.x * 256; i0 < n; i0 += (unsigned long long)gridDim.x * 256) {
    const unsigned long long i = i0 + threadIdx.x;
    int digit = -1;
    if (i < n) {
      const unsigned long long key = keys[i];
      if ((key & hi) == (pre & hi)) digit = (int)((key >> shift) & 255);
    }
    const unsigned peers = __match_any_sync(0xffffffffu, digit);
    if (digit >= 0 && lane == __ffs(peers) - 1) atomicAdd(&hs[digit], (unsigned)__popc(peers));
  }
  __syncthreads();
  if (hs[threadIdx.x]) atomicAdd(&dist->hist[c][threadIdx.x], (unsigned long long)hs[threadIdx.x]);
}

// the digit holding the wanted rank: fix it in the prefix, keep the rank inside it, clear the histogram
__global__ void __launch_bounds__(256) select_digit_kernel(EvalDist* __restrict__ dist, int shift) {
  __shared__ unsigned long long hs[256];
  const int c = blockIdx.x + 1;
  if (dist->list_n[c] == 0) return;
  hs[threadIdx.x] = dist->hist[c][threadIdx.x];
  dist->hist[c][threadIdx.x] = 0;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long r = dist->rank[c];
    int d = 0;
    for (; d < 255 && r >= hs[d]; ++d) r -= hs[d];
    dist->rank[c] = r;
    dist->prefix[c] |= (unsigned long long)d << shift;
  }
}

// the order statistic after the selected one: keys <= it and the smallest key above it
__global__ void __launch_bounds__(256) select_next_kernel(const double* __restrict__ list, EvalDist* __restrict__ dist) {
  __shared__ unsigned long long s_le[8], s_min[8];
  const int c = blockIdx.y + 1;
  const unsigned long long n = dist->list_n[c];
  if (n == 0) return;
  const unsigned long long sel = dist->prefix[c];
  const unsigned long long* __restrict__ keys = reinterpret_cast<const unsigned long long*>(list + dist->list_off[c]);
  unsigned long long le = 0, mn = ~0ull;
  for (unsigned long long i = (unsigned long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * 256) {
    const unsigned long long key = keys[i];
    if (key <= sel) ++le;
    else mn = key < mn ? key : mn;
  }
  for (int o = 16; o; o >>= 1) {
    le += __shfl_xor_sync(0xffffffffu, le, o);
    const unsigned long long m2 = __shfl_xor_sync(0xffffffffu, mn, o);
    mn = m2 < mn ? m2 : mn;
  }
  if ((threadIdx.x & 31) == 0) { s_le[threadIdx.x >> 5] = le; s_min[threadIdx.x >> 5] = mn; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { le += s_le[w]; mn = s_min[w] < mn ? s_min[w] : mn; }
    if (le) atomicAdd(&dist->le[c], le);
    if (mn != ~0ull) atomicMin(&dist->gt_min[c], mn);
  }
}

static double key_value(unsigned long long k) {
  double d;
  memcpy(&d, &k, sizeof(d));
  return d;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

int evaluate_segmentation(sc_ctx* ctx, const uint8_t* seg, const uint8_t* ref, const int32_t* dims, const double* spacing,
                          sc_structure_metrics* metrics, int64_t* confusion, cudaStream_t st) {
  const int X = dims[0], Y = dims[1], Z = dims[2];
  const int64_t total = (int64_t)X * Y * Z;
  const size_t o_counts = align256((size_t)total), o_dist = o_counts + align256(sizeof(EvalCounts));
  SC_TRY(ensure_ws(ctx->ws_train, o_dist + sizeof(EvalDist)));
  char* wbase = reinterpret_cast<char*>(ctx->ws_train.ptr);
  uint8_t* surf = reinterpret_cast<uint8_t*>(wbase);
  EvalCounts* d_counts = reinterpret_cast<EvalCounts*>(wbase + o_counts);
  EvalDist* d_dist = reinterpret_cast<EvalDist*>(wbase + o_dist);
  {
    ProfScope prof(ctx, PC_EVALUATE, st);
    eval_init_kernel<<<1, 256, 0, st>>>(d_counts, d_dist, X, Y, Z);
    const int64_t blocks = (total + 255) / 256;
    const unsigned grid = (unsigned)(blocks < (int64_t)ctx->sm_count * 8 ? blocks : (int64_t)ctx->sm_count * 8);
    eval_surface_kernel<<<grid, 256, 0, st>>>(seg, ref, X, Y, Z, surf, d_counts);
    ctx->launches += 2;
  }
  SC_CUDA(cudaGetLastError());
  EvalCounts hc;
  SC_CUDA(cudaMemcpyAsync(&hc, d_counts, sizeof(hc), cudaMemcpyDeviceToHost, st));
  SC_CUDA(cudaStreamSynchronize(st));
  for (int w = 0; w < 2; ++w)
    SC_CHECK(hc.invalid[w] == 0, SC_ERR_ARG, "sc_evaluate_segmentation: %s holds %llu voxels with a label above 15", w == 0 ? "seg" : "ref",
             (unsigned long long)hc.invalid[w]);

  // per class: counts from the confusion matrix, the distance work only where both structures exist
  int64_t n_seg[16] = {}, n_ref[16] = {};
  for (int r = 0; r < 15; ++r)
    for (int s = 0; s < 15; ++s) {
      n_seg[s] += (int64_t)hc.conf[r * 15 + s];
      n_ref[r] += (int64_t)hc.conf[r * 15 + s];
    }
  unsigned long long list_total = 0, sel[2][16] = {};      // rank | list_off of EvalDist
  unsigned long long* rank = sel[0];
  unsigned long long* list_off = sel[1];
  int64_t max_box = 0;
  double gamma[16] = {};
  bool dist_on[16] = {};
  for (int c = 1; c <= 14; ++c) {
    if (!n_seg[c] || !n_ref[c]) continue;
    dist_on[c] = true;
    const int* bx = hc.box[c];
    const int64_t bv = (int64_t)(bx[1] - bx[0]) * (bx[3] - bx[2]) * (bx[5] - bx[4]);
    max_box = bv > max_box ? bv : max_box;
    list_off[c] = list_total;
    const unsigned long long n = hc.nsurf[0][c] + hc.nsurf[1][c];
    list_total += n;
    // np.percentile(d, 95), method 'linear': virtual index n q + (1 - q) - 1, clipped to [0, n - 1]; interpolation
    // weight = virtual index - its floor (numpy's _compute_virtual_index / _get_indexes / _get_gamma)
    const double q = 0.95, vi = ((double)n * q + (1.0 + q * (1.0 - 1.0 - 1.0))) - 1.0;
    if (vi >= (double)(n - 1)) rank[c] = n - 1;
    else if (vi < 0.0) rank[c] = 0;
    else {
      rank[c] = (unsigned long long)floor(vi);
      gamma[c] = vi - (double)rank[c];
    }
  }
  EvalDist hd;
  memset(&hd, 0, sizeof(hd));
  if (list_total) {
    const size_t o_h = align256((size_t)max_box * 2 * sizeof(int)), o_sv = o_h + align256((size_t)max_box * 2 * sizeof(double));
    const size_t o_sf = o_sv + align256((size_t)max_box * 2 * sizeof(int)), o_sz = o_sf + align256((size_t)max_box * 2 * sizeof(double));
    const size_t o_list = o_sz + align256((size_t)max_box * 2 * sizeof(double));
    SC_TRY(ensure_ws(ctx->ws_eval, o_list + (size_t)list_total * sizeof(double)));
    char* eb = reinterpret_cast<char*>(ctx->ws_eval.ptr);
    int* g = reinterpret_cast<int*>(eb);
    double* h = reinterpret_cast<double*>(eb + o_h);
    int* sv = reinterpret_cast<int*>(eb + o_sv);
    double* sf = reinterpret_cast<double*>(eb + o_sf);
    double* sz = reinterpret_cast<double*>(eb + o_sz);
    double* list = reinterpret_cast<double*>(eb + o_list);
    SC_CUDA(cudaMemcpyAsync(d_dist->rank, sel, sizeof(sel), cudaMemcpyHostToDevice, st));
    ProfScope prof(ctx, PC_EVALUATE, st);
    for (int c = 1; c <= 14; ++c) {
      if (!dist_on[c]) continue;
      const int* bx = hc.box[c];
      const EvalBox b{bx[0], bx[2], bx[4], bx[1] - bx[0], bx[3] - bx[2], bx[5] - bx[4]};
      const int64_t lx = (int64_t)b.by * b.bz, ly = (int64_t)b.bx * b.bz, lz = (int64_t)b.bx * b.by;
      edt_x_kernel<<<dim3((unsigned)((lx + kEdtThreads - 1) / kEdtThreads), 2), kEdtThreads, 0, st>>>(seg, ref, surf, Y, Z, b, c, g);
      edt_y_kernel<<<dim3((unsigned)((ly + kEdtThreads - 1) / kEdtThreads), 2), kEdtThreads, 0, st>>>(g, b, spacing[0], spacing[1], h, sv, sf, sz);
      edt_z_kernel<<<dim3((unsigned)((lz + kEdtThreads - 1) / kEdtThreads), 2), kEdtThreads, 0, st>>>(
          seg, ref, surf, Y, Z, b, c, spacing[2], h, sv, sf, sz, list + list_off[c], d_dist);
      ctx->launches += 3;
    }
    unsigned long long max_n = 0;
    for (int c = 1; c <= 14; ++c) {
      const unsigned long long n = hc.nsurf[0][c] + hc.nsurf[1][c];
      if (dist_on[c] && n > max_n) max_n = n;
    }
    const unsigned long long sb = (max_n + 255) / 256;
    const unsigned sgrid = (unsigned)(sb < (unsigned long long)ctx->sm_count * 2 ? sb : (unsigned long long)ctx->sm_count * 2);
    for (int shift = 56; shift >= 0; shift -= 8) {
      select_hist_kernel<<<dim3(sgrid, 14), 256, 0, st>>>(list, d_dist, shift);
      select_digit_kernel<<<14, 256, 0, st>>>(d_dist, shift);
    }
    select_next_kernel<<<dim3(sgrid, 14), 256, 0, st>>>(list, d_dist);
    ctx->launches += 17;
    SC_CUDA(cudaGetLastError());
  }
  SC_CUDA(cudaMemcpyAsync(&hd, d_dist, offsetof(EvalDist, hist), cudaMemcpyDeviceToHost, st));
  SC_CUDA(cudaStreamSynchronize(st));

  const double nan = NAN;
  sc_structure_metrics out[14];
  for (int c = 1; c <= 14; ++c) {
    sc_structure_metrics& m = out[c - 1];
    m.n_seg = n_seg[c]; m.n_ref = n_ref[c]; m.n_both = (int64_t)hc.conf[c * 15 + c];
    m.dice = n_seg[c] + n_ref[c] ? (double)(2 * m.n_both) / (double)(n_seg[c] + n_ref[c]) : nan;
    m.vol_seg_mm3 = (double)n_seg[c] * spacing[0] * spacing[1] * spacing[2];
    m.vol_ref_mm3 = (double)n_ref[c] * spacing[0] * spacing[1] * spacing[2];
    m.hd_mm = m.hd95_mm = m.assd_mm = nan;
    if (!dist_on[c]) continue;
    SC_CHECK(hd.cnt[c][0] == hc.nsurf[0][c] && hd.cnt[c][1] == hc.nsurf[1][c] && hd.list_n[c] == hc.nsurf[0][c] + hc.nsurf[1][c],
             SC_ERR_STATE, "sc_evaluate_segmentation: internal: class %d sampled %llu + %llu of %llu + %llu surface voxels", c,
             (unsigned long long)hd.cnt[c][0], (unsigned long long)hd.cnt[c][1], (unsigned long long)hc.nsurf[0][c],
             (unsigned long long)hc.nsurf[1][c]);
    const double a = key_value(hd.prefix[c]);
    const double b = rank[c] + 1 < hd.le[c] ? a : key_value(hd.gt_min[c]);
    double p = a;
    if (rank[c] + 1 < hd.list_n[c]) {                        // numpy's _lerp: a + (b - a) t, or b - (b - a)(1 - t) for t >= 0.5
      const double t = gamma[c], diff = b - a;
      p = t >= 0.5 ? b - diff * (1.0 - t) : a + diff * t;
    }
    m.hd_mm = fmax(key_value(hd.max[c][0]), key_value(hd.max[c][1]));
    m.hd95_mm = p;
    m.assd_mm = (hd.sum[c][0] / (double)hd.cnt[c][0] + hd.sum[c][1] / (double)hd.cnt[c][1]) / 2.0;
  }
  memcpy(metrics, out, sizeof(out));
  if (confusion)
    for (int i = 0; i < 225; ++i) confusion[i] = (int64_t)hc.conf[i];
  return SC_OK;
}

}  // namespace sc
