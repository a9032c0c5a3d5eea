// tcgen05 / TMEM / TMA back-end of the dense-layer / implicit-GEMM problem (sm_100a).
//
//   C[m, n] = prelu( sum_tap sum_k A[pixel m shifted by tap, k] * W[n, tap*kc + k] + bias[n] )
//
// used for d1 (as a 3x3 dilation-4 conv over the NHWC-64 conv5 map), FC1 and fc_2
// (reference: DenseLayer + PReLU at cnn_cort/nets.py:179-180, 217-218, 227-228).
//
// Precision: single-pass TF32 / fp16 misses the 1e-3 softmax tolerance on unsaturated inputs
// (measured: 1.4e-3), so the product is the three-MMA split  xh*wh + xh*wl + xl*wh  of bf16 pairs
// (x = xh + xl to ~2^-17, kind::f16 with fp32 accumulation in TMEM; oracle emulation: 1.8e-5).
// Activations and weights are stored per 64-wide k block as 64 bf16 hi | 64 bf16 lo, i.e. exactly
// the bytes of the fp32 row, so one 128 B swizzle row holds one block half.
//
// Two kernels share this file:
//   gemm_tc_pair_kernel        CTA pairs (cta_group::2, M = 256): tiles of >= 128 columns -- d1, FC1 (+ atlas prior
//                              columns), fc_2 (+ out_layer, softmax and argmax in its epilogue), the dense layers of the
//                              training step: the hot ones
//   gemm_tc_persistent_kernel  one persistent CTA per SM (M = 128): narrow layers
// Both: warp 0 = TMA producer (per k block A hi, A lo as 4-D boxes of 64 bf16 x 128 pixels with the tap shift applied to
// the pixel / line / plane coordinates and zero fill outside, W hi, W lo as 2-D boxes), warp 1 = converged MMA issue
// (12 x tcgen05.mma K=16 per k block), the other warps = epilogue (tcgen05.ld -> scale / bias / PReLU -> plain fp32 or
// split bf16 rows); two TMEM accumulators so that the epilogue of tile i overlaps the main loop of tile i + 1.
// (conv2..conv5 live in conv_sweep.cu.)
#include "tc_common.cuh"

namespace sc {

__device__ __forceinline__ void tmem_ld16(uint32_t (&r)[16], uint32_t taddr) {   // 32 lanes x 16 consecutive 32-bit columns
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;                    // logical k per block (64 bf16 = one 128 B swizzle row)
constexpr int TC_A_HALF = TC_BM * 128;       // bytes of the hi (or lo) half of an A stage

struct TcArgs {
  int kpt;            // k-blocks per tap (kc / 64)
  int nkb;            // total k-blocks
  int stages;
  int bn;             // tile columns (multiple of 16, <= 192)
  int nt, mt;         // tiles along n, along m (per line)
  int Y;              // lines per plane
  int M;              // rows per line
  int n_store, npad, c_col0;
  int a_y0, a_z0;     // coordinate offsets of line / plane in the A tensor map
  int a_swap;         // tensor-map dimension order (k, pixel, plane, line): swap the last two coordinates
  int tap_dx[9], tap_dy[9], tap_dz[9];
  float* C;
  long long ldc, c_ys, c_zs;
  const float* bias;
  const float* alpha;
  const float* scale;
  int out_split;
  // persistent variant
  long long num_tiles;
  int epi_warps;      // epilogue warps (4, 8 or 16)
  int last_ksteps;    // 16-wide k-steps issued in the LAST k block (dense layers: the K padding beyond the real fan-in is skipped)
  unsigned long long* dbg;   // optional per-CTA cycle counters [8] (sc_set_option "tc_timing"): where each role waits
  const int* rowmap;  // pair kernel, split stores: C row of dense row r = rowmap[r] (skip when < 0); ldc / c_ys / c_zs then count ROWS
  const int* rowvox;  // pair kernel, atlas epilogue: slab row of compact row m
  long long crow_ld;  // floats per C row in rowmap mode
  int n_mma;          // pair kernel: columns the MMAs have to produce (real N rounded to 16): the last n-tile issues narrower MMAs
  const unsigned char* tile_on;   // pair kernel: tile t is computed only if tile_on[t] != 0 (row map: no candidate row in it)
  const float* atlas; // pair kernel: atlas prior volume [X][Y][Z][15] -> output columns 540..575 (see GemmProblem::atlas)
  OutGeo ageo;
  SoftmaxOut sm;      // pair kernel, fc_2 with the out_layer epilogue (FUSED_OUT): where the softmax / argmax results go
  const float* out_w; // FUSED_OUT: out_layer weights [270][16] and bias [16], fp32
  const float* out_b;
  float* mc_acc;      // MC_ACC: per-row Monte-Carlo dropout accumulator [M][16] (see GemmProblem::mc_acc)
  int mc_first;
};

// fused out_layer (FUSED_OUT): the 16 epilogue warps' store-transpose area is free and holds the out_layer weights (rows padded
// to 272 with zeros: fc_2's last chunk ends at column 271), the bias, and the logit partials of column groups 1..3
constexpr int kOutWFloats = kH2Ld * 16;
constexpr int kOutPartFloats = 3 * 15 * TC_BM;          // [group - 1][class][row of the CTA]
static_assert((kOutWFloats + 16 + kOutPartFloats) * 4 <= 16 * 2560, "fused out_layer scratch exceeds the store-transpose area");

// ---------------------------------------------------------------------------------------------------
// Persistent kernel: one CTA per SM walks the tile list (tile = blockIdx.x + i * gridDim.x).
//   * shared-memory ring of A + W stages fed by TMA, decoupled from the MMA warp by full/empty mbarriers
//   * two TMEM accumulators (columns 0.. and 256..): the epilogue of tile i overlaps the main loop of tile i+1
// ---------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(576, 1)
gemm_tc_persistent_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024 B aligned, still a shared-space pointer
  const int b_half = a.bn * 128;
  const int w_block = 2 * b_half;                               // hi | lo of one 64-wide k block of W
  const int stage_bytes = 2 * TC_A_HALF + w_block;
  uint8_t* sStage = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStage + a.stages * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + a.stages;
  uint64_t* tfull = bars + 2 * a.stages;     // [2] accumulator ready
  uint64_t* tempty = tfull + 2;              // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* s_const = reinterpret_cast<float*>(tmem_slot + 4);   // [2 buffers][bias bn | alpha bn | scale bn], 16 B aligned (float4 loads)
  uint8_t* s_stage = reinterpret_cast<uint8_t*>(s_const + 2 * 3 * a.bn);   // [epilogue warps][32 rows][80 B] store-transpose tiles

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], (blockDim.x >> 5) - 2); }
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

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB)) : "memory");
      uint32_t it = 0;   // global stage-use counter
      long long dbg_acc[1] = {0};
      const long long tstart = a.dbg ? clock64() : 0;
      for (long long t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
        long long r = t;
        const int n_tile = (int)(r % a.nt); r /= a.nt;
        const int m_tile = (int)(r % a.mt); r /= a.mt;
        const int y = (int)(r % a.Y);
        const int z = (int)(r / a.Y);
        const int m0 = m_tile * TC_BM, n0 = n_tile * a.bn;
        for (int kb = 0; kb < a.nkb; ++kb, ++it) {
          const int s = it % a.stages;
          const uint32_t use = it / a.stages;
          if (use > 0) {
            const long long c0 = a.dbg ? clock64() : 0;
            mbar_wait(&empty[s], (use - 1) & 1);
            if (a.dbg) dbg_acc[0] += clock64() - c0;
          }
          mbar_expect_tx(&full[s], (uint32_t)stage_bytes);
          uint8_t* sp = sStage + s * stage_bytes;
          const int tap = kb / a.kpt, ka = (kb - tap * a.kpt) * 2 * TC_BK;
          const int px = m0 + a.tap_dx[tap], ln = y + a.a_y0 + a.tap_dy[tap], pl = z + a.a_z0 + a.tap_dz[tap];
          tma_load_4d(&mapA, &full[s], sp, ka, px, a.a_swap ? pl : ln, a.a_swap ? ln : pl);
          tma_load_4d(&mapA, &full[s], sp + TC_A_HALF, ka + TC_BK, px, a.a_swap ? pl : ln, a.a_swap ? ln : pl);
          tma_load_2d(&mapB, &full[s], sp + 2 * TC_A_HALF, kb * 2 * TC_BK, n0);
          tma_load_2d(&mapB, &full[s], sp + 2 * TC_A_HALF + b_half, kb * 2 * TC_BK + TC_BK, n0);
        }
      }
      if (a.dbg) { a.dbg[blockIdx.x * 8 + 0] = (unsigned long long)dbg_acc[0]; a.dbg[blockIdx.x * 8 + 1] = (unsigned long long)(clock64() - tstart); }
    }
    __syncwarp();
  } else if (warp == 1) {
    // whole warp converged; one elected lane issues (see umma_bf16_elect)
    const uint32_t leader = elect_one();
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(a.bn >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    const uint32_t sStage_u = smem_u32(sStage);
    uint32_t it = 0, ti = 0;
    long long w_full = 0, w_tempty = 0;
    const long long tstart = a.dbg ? clock64() : 0;
    for (long long t = blockIdx.x; t < a.num_tiles; t += gridDim.x, ++ti) {
      const uint32_t b = ti & 1, buse = ti >> 1;
      long long c0 = a.dbg ? clock64() : 0;
      mbar_wait(&tempty[b], (buse & 1) ^ 1);                    // accumulator b drained by the epilogue
      if (a.dbg) w_tempty += clock64() - c0;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t acc = tmem_base + b * 256;
      for (int kb = 0; kb < a.nkb; ++kb, ++it) {
        const int s = it % a.stages;
        c0 = a.dbg ? clock64() : 0;
        mbar_wait(&full[s], (it / a.stages) & 1);
        if (a.dbg) w_full += clock64() - c0;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sp = sStage_u + s * stage_bytes;
        const uint64_t ah = umma_desc(sp), al = umma_desc(sp + TC_A_HALF);
        const uint64_t wh = umma_desc(sp + 2 * TC_A_HALF), wl = umma_desc(sp + 2 * TC_A_HALF + b_half);
#pragma unroll
        for (int j = 0; j < 4; ++j) {   // 4 x K=16 bf16 (32 B) inside the 128 B swizzle row; small terms first
          const uint64_t o = (uint64_t)(j * 2);
          umma_bf16_elect(acc, al + o, wh + o, idesc, (kb | j) != 0, leader);
          umma_bf16_elect(acc, ah + o, wl + o, idesc, 1, leader);
          umma_bf16_elect(acc, ah + o, wh + o, idesc, 1, leader);
        }
        if (leader) umma_commit(&empty[s]);
        __syncwarp();
      }
      if (leader) umma_commit(&tfull[b]);
      __syncwarp();
    }
    if (a.dbg && leader) {
      a.dbg[blockIdx.x * 8 + 2] = (unsigned long long)w_full; a.dbg[blockIdx.x * 8 + 3] = (unsigned long long)w_tempty;
      a.dbg[blockIdx.x * 8 + 4] = (unsigned long long)(clock64() - tstart);
    }
  } else {
    // 4*G epilogue warps: warp w reads TMEM lanes of quarter w%4 (hardware rule) and every G-th 16-column chunk.
    // Several warps per scheduler hide the dependent-issue latency a single epilogue warp would expose.
    const int q = warp & 3;
    const int nepi = (blockDim.x >> 5) - 2, G = nepi >> 2, grp = (warp - 2) >> 2;
    const int epi_threads = nepi * 32;
    uint32_t ti = 0;
    long long w_tfull = 0;
    const long long tstart = a.dbg ? clock64() : 0;
    for (long long t = blockIdx.x; t < a.num_tiles; t += gridDim.x, ++ti) {
      long long r = t;
      const int n_tile = (int)(r % a.nt); r /= a.nt;
      const int m_tile = (int)(r % a.mt); r /= a.mt;
      const int y = (int)(r % a.Y);
      const int z = (int)(r / a.Y);
      const int m0 = m_tile * TC_BM, n0 = n_tile * a.bn;
      const uint32_t b = ti & 1, buse = ti >> 1;
      // this tile's epilogue constants -> shared memory (buffer b; its previous readers finished two tiles ago)
      float* cb = s_const + b * 3 * a.bn;
      if (ti < 2 || a.nt > 1) {
        for (int i = threadIdx.x - 64; i < a.bn; i += epi_threads) {
          const int nn = n0 + i;
          const bool ok = nn < a.npad;
          cb[i] = ok ? __ldg(a.bias + nn) : 0.f;
          cb[a.bn + i] = ok ? __ldg(a.alpha + nn) : 1.f;
          cb[2 * a.bn + i] = (a.scale && ok) ? __ldg(a.scale + nn) : 1.f;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
      }
      const long long c0w = a.dbg ? clock64() : 0;
      mbar_wait(&tfull[b], buse & 1);
      if (a.dbg) w_tfull += clock64() - c0w;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // Each thread owns one accumulator row, but a row-per-thread store touches 32 sectors per instruction.
      // A 2.5 KB per-warp shared tile transposes every 16-column chunk so that adjacent lanes write adjacent
      // 16 B pieces: every global store instruction fills whole 32 B sectors.
      float* ctile = a.C + (long long)z * a.c_zs + (long long)y * a.c_ys;
      const int mw = m0 + q * 32;                       // first row of this warp
      uint8_t* stg = s_stage + (warp - 2) * 2560;
      uint8_t* mine = stg + lane * 80;
      for (int c0 = grp * 16; c0 < a.bn; c0 += 16 * G) {
        uint32_t rr[16];
        const uint32_t taddr = tmem_base + b * 256 + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(rr[0]), "=r"(rr[1]), "=r"(rr[2]), "=r"(rr[3]), "=r"(rr[4]), "=r"(rr[5]), "=r"(rr[6]), "=r"(rr[7]), "=r"(rr[8]),
              "=r"(rr[9]), "=r"(rr[10]), "=r"(rr[11]), "=r"(rr[12]), "=r"(rr[13]), "=r"(rr[14]), "=r"(rr[15])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (n0 + c0 >= a.n_store) continue;             // warp-uniform
        float v[16];
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const float4 bi = *reinterpret_cast<const float4*>(cb + c0 + 4 * k4);
          const float4 al = *reinterpret_cast<const float4*>(cb + a.bn + c0 + 4 * k4);
          const float4 sc_ = *reinterpret_cast<const float4*>(cb + 2 * a.bn + c0 + 4 * k4);
          v[4 * k4 + 0] = prelu(fmaf(__uint_as_float(rr[4 * k4 + 0]), sc_.x, bi.x), al.x);
          v[4 * k4 + 1] = prelu(fmaf(__uint_as_float(rr[4 * k4 + 1]), sc_.y, bi.y), al.y);
          v[4 * k4 + 2] = prelu(fmaf(__uint_as_float(rr[4 * k4 + 2]), sc_.z, bi.z), al.z);
          v[4 * k4 + 3] = prelu(fmaf(__uint_as_float(rr[4 * k4 + 3]), sc_.w, bi.w), al.w);
        }
        const int ncol = a.c_col0 + n0 + c0;            // multiple of 16
        if (a.out_split) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
          *reinterpret_cast<uint4*>(mine) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(mine + 16) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
          *reinterpret_cast<uint4*>(mine + 32) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(mine + 48) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
          __syncwarp();
          const int boff = (ncol >> 6) * 128 + (ncol & 63);   // bf16 offset of the hi piece inside the row
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int half = i >> 1, row = (i & 1) * 16 + (lane >> 1), part = lane & 1;
            const uint4 d = *reinterpret_cast<const uint4*>(stg + row * 80 + half * 32 + part * 16);
            if (mw + row < a.M) {
              __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(ctile + (long long)(mw + row) * a.ldc) + boff + half * 64 + part * 8;
              *reinterpret_cast<uint4*>(dst) = d;
            }
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(mine + 16 * k) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = i * 8 + (lane >> 2), part = lane & 3;
            const float4 d = *reinterpret_cast<const float4*>(stg + row * 80 + part * 16);
            if (mw + row < a.M) *reinterpret_cast<float4*>(ctile + (long long)(mw + row) * a.ldc + ncol + part * 4) = d;
          }
        }
        __syncwarp();
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[b]);
    }
    if (a.dbg && threadIdx.x == 64) {
      a.dbg[blockIdx.x * 8 + 5] = (unsigned long long)w_tfull; a.dbg[blockIdx.x * 8 + 6] = (unsigned long long)(clock64() - tstart);
      a.dbg[blockIdx.x * 8 + 7] = ti;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2) for the wide streaming-weight tiles (d1, FC1, fc_2): a cluster of two CTAs on
// an SM pair computes a 256-row tile.  Each CTA loads its own 128 rows of A but only HALF of the weight block
// (bn/2 rows), so the weight bytes every SM has to ingest per MMA halve and a third pipeline stage fits.
//   * both producers signal the LEADER's full barrier (cta_group::2 TMA, peer bit cleared in the barrier address)
//   * the leader's MMA warp issues tcgen05.mma.cta_group::2 (M = 256) and multicasts its commits to both CTAs
//   * every CTA's epilogue warps drain their own TMEM half and arrive on the leader's tempty barrier (remote arrive)
// ---------------------------------------------------------------------------------------------------
// MC_ACC (with FUSED_OUT): one Monte-Carlo dropout pass -- the softmax of row m and its sum_c p_c ln p_c are added to
// mc_acc[m * 16 ..] (stored by the first pass) in pass order, instead of being scattered into the volume
template <bool FUSED_OUT, bool MC_ACC = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(576, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int hb = a.bn >> 1;                               // weight rows held by this CTA
  const int b_half = hb * 128;                            // bytes of its hi (or lo) weight half-block
  const int stage_bytes = 2 * TC_A_HALF + 2 * b_half;
  uint8_t* sStage = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStage + a.stages * stage_bytes);
  uint64_t* full = bars;                                  // used in the leader only (both producers signal it)
  uint64_t* empty = bars + a.stages;                      // per CTA, arrived by the leader's multicast commit
  uint64_t* tfull = bars + 2 * a.stages;                  // [2] per CTA
  uint64_t* tempty = tfull + 2;                           // [2] leader only: both CTAs' epilogue warps arrive
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  // float4 loads of the constants need 16 B alignment; plain pointer arithmetic on `smem` keeps the shared address space (LDS / STS)
  float* s_const = reinterpret_cast<float*>(smem + (((size_t)a.stages * stage_bytes + (2 * a.stages + 4) * 8 + 16 + 15) & ~(size_t)15));
  uint8_t* s_stage = reinterpret_cast<uint8_t*>(s_const + (a.nt > 2 ? a.nt : 2) * 3 * a.bn);   // constants of every n-tile (<= 4) stay resident

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();                 // position inside the CTA pair; rank 0 leads
  const int nepi = (blockDim.x >> 5) - 2;
  // every pair walks the flat tile list in work units of `per` consecutive tiles: one tile, or with the fused out_layer all n-tiles
  // of a 256-row block, so that one CTA pair's epilogue sees every fc_2 output of its rows
  const int pair = (int)(blockIdx.x >> 1), npairs = (int)(gridDim.x >> 1);   // (the host keeps the tile count below 2^31)
  const int per = FUSED_OUT ? a.nt : 1;
  const int units = (int)(a.num_tiles / per);

  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 2 * nepi); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB)) : "memory");
      uint32_t it = 0;
      long long w_empty = 0;
      const long long tstart = a.dbg ? clock64() : 0;
      for (int u = pair; u < units; u += npairs)
      for (int jt = 0; jt < per; ++jt) {
        const int t = u * per + jt;
        if (a.tile_on && !a.tile_on[t]) continue;
        long long r = t;
        const int n_tile = (int)(r % a.nt); r /= a.nt;
        const int m_tile = (int)(r % a.mt); r /= a.mt;
        const int y = (int)(r % a.Y);
        const int z = (int)(r / a.Y);
        const int bnj = min(a.bn, a.n_mma - n_tile * a.bn);            // MMA width of this n-tile (the last one may be narrower)
        const int m0 = m_tile * 256 + (int)rank * TC_BM, n0 = n_tile * a.bn + (int)rank * (bnj >> 1);
        for (int kb = 0; kb < a.nkb; ++kb, ++it) {
          const int s = it % a.stages;
          const uint32_t use = it / a.stages;
          if (use > 0) {
            const long long c0 = a.dbg ? clock64() : 0;
            mbar_wait(&empty[s], (use - 1) & 1);
            if (a.dbg) w_empty += clock64() - c0;
          }
          uint8_t* sp = sStage + s * stage_bytes;
          const int tap = kb / a.kpt, ka = (kb - tap * a.kpt) * 2 * TC_BK;
          const int px = m0 + a.tap_dx[tap], ln = y + a.a_y0 + a.tap_dy[tap], pl = z + a.a_z0 + a.tap_dz[tap];
          const uint32_t lbar = smem_u32(&full[s]) & 0xFEFFFFFFu;    // the leader's barrier (peer bit cleared)
          if (rank == 0) mbar_expect_tx(&full[s], (uint32_t)(2 * stage_bytes));   // both CTAs' bytes land on it
          tma_load_4d_2sm(&mapA, lbar, sp, ka, px, a.a_swap ? pl : ln, a.a_swap ? ln : pl);
          tma_load_4d_2sm(&mapA, lbar, sp + TC_A_HALF, ka + TC_BK, px, a.a_swap ? pl : ln, a.a_swap ? ln : pl);
          tma_load_2d_2sm(&mapB, lbar, sp + 2 * TC_A_HALF, kb * 2 * TC_BK, n0);
          tma_load_2d_2sm(&mapB, lbar, sp + 2 * TC_A_HALF + b_half, kb * 2 * TC_BK + TC_BK, n0);
        }
      }
      if (a.dbg && rank == 0) { a.dbg[pair * 8 + 0] = (unsigned long long)w_empty; a.dbg[pair * 8 + 1] = (unsigned long long)(clock64() - tstart); }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (rank == 0) {
      const uint32_t leader = elect_one();
      // instruction descriptor: D=F32, A=B=BF16, K-major, N = bn, M = 256 (two CTAs x 128 rows)
      const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 4) << 24);
      const uint32_t sStage_u = smem_u32(sStage);
      uint32_t it = 0, ti = 0;
      long long w_full = 0, w_tempty = 0;
      const long long tstart = a.dbg ? clock64() : 0;
      for (int u = pair; u < units; u += npairs)
      for (int jt = 0; jt < per; ++jt) {
        const int t = u * per + jt;
        if (a.tile_on && !a.tile_on[t]) continue;
        const uint32_t b = ti & 1, buse = ti >> 1;
        const int bnj = min(a.bn, a.n_mma - (int)(t % a.nt) * a.bn);
        const uint32_t idesc = idesc0 | ((uint32_t)(bnj >> 3) << 17);   // N = bnj (bnj / 2 weight rows from each CTA)
        long long c0 = a.dbg ? clock64() : 0;
        mbar_wait(&tempty[b], (buse & 1) ^ 1);
        if (a.dbg) w_tempty += clock64() - c0;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t acc = tmem_base + b * 256;
        for (int kb = 0; kb < a.nkb; ++kb, ++it) {
          const int s = it % a.stages;
          c0 = a.dbg ? clock64() : 0;
          mbar_wait(&full[s], (it / a.stages) & 1);
          if (a.dbg) w_full += clock64() - c0;
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sp = sStage_u + s * stage_bytes;
          const uint64_t ah = umma_desc(sp), al = umma_desc(sp + TC_A_HALF);
          const uint64_t wh = umma_desc(sp + 2 * TC_A_HALF), wl = umma_desc(sp + 2 * TC_A_HALF + b_half);
          const int nj = kb == a.nkb - 1 ? a.last_ksteps : 4;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint64_t o = (uint64_t)(j * 2);
            const uint32_t on = (leader && j < nj) ? 1u : 0u;
            umma_bf16_2sm_elect(acc, al + o, wh + o, idesc, (kb | j) != 0, on);
            umma_bf16_2sm_elect(acc, ah + o, wl + o, idesc, 1, on);
            umma_bf16_2sm_elect(acc, ah + o, wh + o, idesc, 1, on);
          }
          if (leader) umma_commit_2sm(&empty[s]);
          __syncwarp();
        }
        if (leader) umma_commit_2sm(&tfull[b]);
        __syncwarp();
        ++ti;
      }
      if (a.dbg && leader) {
        a.dbg[pair * 8 + 2] = (unsigned long long)w_full; a.dbg[pair * 8 + 3] = (unsigned long long)w_tempty;
        a.dbg[pair * 8 + 4] = (unsigned long long)(clock64() - tstart);
      }
    }
  } else {
    const int q = warp & 3;
    const int G = nepi >> 2, grp = (warp - 2) >> 2;
    const int epi_threads = nepi * 32;
    uint32_t ti = 0;
    long long w_tfull = 0;
    // epilogue constants (bias / BN shift, PReLU slope, BN scale) of all n-tiles: shared memory, once per kernel
    for (int i = threadIdx.x - 64; i < a.nt * a.bn; i += epi_threads) {
      const int j = i / a.bn, c = i - j * a.bn, nn = i;
      const bool ok = nn < a.npad;
      float* cbw = s_const + j * 3 * a.bn;
      cbw[c] = ok ? __ldg(a.bias + nn) : 0.f;
      cbw[a.bn + c] = ok ? __ldg(a.alpha + nn) : 1.f;
      cbw[2 * a.bn + c] = (a.scale && ok) ? __ldg(a.scale + nn) : 1.f;
    }
    float* s_ow = reinterpret_cast<float*>(s_stage);    // FUSED_OUT: see kOutWFloats
    float* s_ob = s_ow + kOutWFloats;
    float* s_part = s_ob + 16;
    if (FUSED_OUT) {
      for (int i = threadIdx.x - 64; i < kOutWFloats + 16; i += epi_threads)
        s_ow[i] = i < 270 * 16 ? __ldg(a.out_w + i) : (i >= kOutWFloats ? __ldg(a.out_b + i - kOutWFloats) : 0.f);
    }
    asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
    float logit[15];                                      // FUSED_OUT: this thread's share of its row's out_layer logits
    const long long tstart = a.dbg ? clock64() : 0;
    for (int u = pair; u < units; u += npairs)
    for (int jt = 0; jt < per; ++jt) {
      const int t = u * per + jt;
      if (a.tile_on && !a.tile_on[t]) continue;
      long long r = t;
      const int n_tile = (int)(r % a.nt); r /= a.nt;
      const int m_tile = (int)(r % a.mt); r /= a.mt;
      const int y = (int)(r % a.Y);
      const int z = (int)(r / a.Y);
      const int m0 = m_tile * 256 + (int)rank * TC_BM, n0 = n_tile * a.bn;
      const uint32_t b = ti & 1, buse = ti >> 1;
      const float* cb = s_const + n_tile * 3 * a.bn;     // loaded once before the tile loop
      const long long c0w = a.dbg ? clock64() : 0;
      mbar_wait(&tfull[b], buse & 1);
      if (a.dbg) w_tfull += clock64() - c0w;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      float* ctile = a.C + (long long)z * a.c_zs + (long long)y * a.c_ys;
      const int mw = m0 + q * 32;
      uint8_t* stg = s_stage + (warp - 2) * 2560;
      uint8_t* mine = stg + lane * 80;
      if (FUSED_OUT) {
        // One 16-column chunk at a time: bias / PReLU, then the out_layer as fp32 FMAs into this thread's logit partials (the
        // weight rows are broadcast reads).  Nothing is stored.  The accumulator goes back to the MMA warp after the last chunk;
        // this epilogue is short next to the MMAs of the next tile, which run in the other accumulator meanwhile.
        if (jt == 0) {
#pragma unroll
          for (int c = 0; c < 15; ++c) logit[c] = 0.f;
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c0 = grp * 16 + i * 16 * G;
          if (c0 >= a.bn || n0 + c0 >= a.n_store) continue;     // warp-uniform
          uint32_t r[16];
          tmem_ld16(r, tmem_base + b * 256 + ((uint32_t)(q * 32) << 16) + (uint32_t)c0);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          const float4* w4 = reinterpret_cast<const float4*>(s_ow + (n0 + c0) * 16);
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            const float x = prelu(fmaf(__uint_as_float(r[k]), cb[2 * a.bn + c0 + k], cb[c0 + k]), cb[a.bn + c0 + k]);
            const float4 w0 = w4[4 * k], w1 = w4[4 * k + 1], w2 = w4[4 * k + 2], w3 = w4[4 * k + 3];
            logit[0] = fmaf(x, w0.x, logit[0]); logit[1] = fmaf(x, w0.y, logit[1]);
            logit[2] = fmaf(x, w0.z, logit[2]); logit[3] = fmaf(x, w0.w, logit[3]);
            logit[4] = fmaf(x, w1.x, logit[4]); logit[5] = fmaf(x, w1.y, logit[5]);
            logit[6] = fmaf(x, w1.z, logit[6]); logit[7] = fmaf(x, w1.w, logit[7]);
            logit[8] = fmaf(x, w2.x, logit[8]); logit[9] = fmaf(x, w2.y, logit[9]);
            logit[10] = fmaf(x, w2.z, logit[10]); logit[11] = fmaf(x, w2.w, logit[11]);
            logit[12] = fmaf(x, w3.x, logit[12]); logit[13] = fmaf(x, w3.y, logit[13]);
            logit[14] = fmaf(x, w3.z, logit[14]);
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(&tempty[b], 0);
        ++ti;
        if (jt == per - 1) {
          // the block's last n-tile: column groups 1..3 hand their logit partials to group 0 through shared memory; the second
          // barrier keeps the next block's partials from overwriting these before group 0 has read them
          const int crow = q * 32 + lane;
          if (grp > 0) {
#pragma unroll
            for (int c = 0; c < 15; ++c) s_part[((grp - 1) * 15 + c) * TC_BM + crow] = logit[c];
          }
          asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
          if (grp == 0) {
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
              for (int c = 0; c < 15; ++c) logit[c] += s_part[(g * 15 + c) * TC_BM + crow];
          }
          asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
          long long m = (long long)mw + lane;
          bool ok = grp == 0 && m < a.M;
          if (MC_ACC) {
            if (ok) {
#pragma unroll
              for (int c = 0; c < 15; ++c) logit[c] += s_ob[c];
              softmax15(logit);
              float4* acc = reinterpret_cast<float4*>(a.mc_acc + m * 16);
              const float4 v[4] = {make_float4(logit[0], logit[1], logit[2], logit[3]), make_float4(logit[4], logit[5], logit[6], logit[7]),
                                   make_float4(logit[8], logit[9], logit[10], logit[11]),
                                   make_float4(logit[12], logit[13], logit[14], plogp15(logit))};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                float4 r = v[i];
                if (!a.mc_first) {
                  const float4 o = acc[i];
                  r.x += o.x; r.y += o.y; r.z += o.z; r.w += o.w;
                }
                acc[i] = r;
              }
            }
            continue;
          }
          if (ok && a.sm.rowvox) m = __ldg(a.sm.rowvox + m);      // compact row -> row of the dense slab
          long long o = m;
          if (ok && a.sm.use_geo) {
            const long long plane = (long long)a.sm.geo.by * a.sm.geo.bz;
            const int ix = (int)(m / plane);
            const int rem = (int)(m - (long long)ix * plane);
            const int iy = rem / a.sm.geo.bz, iz = rem - iy * a.sm.geo.bz;
            o = ((long long)(a.sm.geo.x0 + ix) * a.sm.geo.Y + (a.sm.geo.y0 + iy)) * a.sm.geo.Z + (a.sm.geo.z0 + iz);
            if (a.sm.mask && a.sm.mask[o] == 0) ok = false;
          }
          if (ok) {
#pragma unroll
            for (int c = 0; c < 15; ++c) logit[c] += s_ob[c];
            softmax_store(logit, o, a.sm.proba, a.sm.label32, a.sm.label8);
          }
        }
        continue;
      }
      // The warp's (up to three) 16-column chunks of the accumulator go to registers first; the accumulator is handed back
      // to the MMA warp right after that, so the arithmetic and the stores of this tile overlap the MMAs of the tile after next.
      uint32_t rr[3][16];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const int c0 = grp * 16 + i * 16 * G;
        if (c0 < a.bn) tmem_ld16(rr[i], tmem_base + b * 256 + ((uint32_t)(q * 32) << 16) + (uint32_t)c0);
      }
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive_cta(&tempty[b], 0);     // the leader's MMA warp owns the accumulator hand-off
      // destination row of this lane's accumulator row (the transposed stores below fetch it by shuffle)
      float* myrow = nullptr;
      if (a.out_split && mw + lane < a.M) {
        myrow = ctile + (long long)(mw + lane) * a.ldc;
        if (a.rowmap) {        // candidate compaction: strides count rows, the map gives the compact C row (or -1)
          const int cr = __ldg(a.rowmap + ((long long)z * a.c_zs + (long long)y * a.c_ys + (long long)(mw + lane) * a.ldc));
          myrow = cr < 0 ? nullptr : a.C + (long long)cr * a.crow_ld;
        }
      }
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const int c0 = grp * 16 + i * 16 * G;
        if (c0 >= a.bn || n0 + c0 >= a.n_store) continue;     // warp-uniform
        if (n0 + c0 >= a.n_mma) {                      // no MMA produced these columns (atlas / zero padding of the row)
#pragma unroll
          for (int kk = 0; kk < 16; ++kk) rr[i][kk] = 0u;
        }
        float v[16];
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const float4 bi = *reinterpret_cast<const float4*>(cb + c0 + 4 * k4);
          const float4 al = *reinterpret_cast<const float4*>(cb + a.bn + c0 + 4 * k4);
          if (a.scale) {
            const float4 sc_ = *reinterpret_cast<const float4*>(cb + 2 * a.bn + c0 + 4 * k4);
            v[4 * k4 + 0] = prelu(fmaf(__uint_as_float(rr[i][4 * k4 + 0]), sc_.x, bi.x), al.x);
            v[4 * k4 + 1] = prelu(fmaf(__uint_as_float(rr[i][4 * k4 + 1]), sc_.y, bi.y), al.y);
            v[4 * k4 + 2] = prelu(fmaf(__uint_as_float(rr[i][4 * k4 + 2]), sc_.z, bi.z), al.z);
            v[4 * k4 + 3] = prelu(fmaf(__uint_as_float(rr[i][4 * k4 + 3]), sc_.w, bi.w), al.w);
          } else {
            v[4 * k4 + 0] = prelu(__uint_as_float(rr[i][4 * k4 + 0]) + bi.x, al.x);
            v[4 * k4 + 1] = prelu(__uint_as_float(rr[i][4 * k4 + 1]) + bi.y, al.y);
            v[4 * k4 + 2] = prelu(__uint_as_float(rr[i][4 * k4 + 2]) + bi.z, al.z);
            v[4 * k4 + 3] = prelu(__uint_as_float(rr[i][4 * k4 + 3]) + bi.w, al.w);
          }
        }
        const int ncol = a.c_col0 + n0 + c0;
        if (a.atlas && (ncol == 528 || ncol == 544)) {
          // atlas prior of this thread's row (cnn_cort/base.py:387-394): atlas[x,y,z,:], all-zero rows become one-hot
          // background; the float32 sum follows numpy's pairwise order.  Columns 540..554 of the h1 row.
          long long mrow = (long long)mw + lane;
          float at[15];
          if (mrow < a.M) {
            if (a.rowvox) mrow = __ldg(a.rowvox + mrow);          // compact row -> row of the dense slab
            const long long plane = (long long)a.ageo.by * a.ageo.bz;
            const int ix = (int)(mrow / plane);
            const int rem = (int)(mrow - (long long)ix * plane);
            const int iy = rem / a.ageo.bz, iz = rem - iy * a.ageo.bz;
            const long long vx = ((long long)(a.ageo.x0 + ix) * a.ageo.Y + (a.ageo.y0 + iy)) * a.ageo.Z + (a.ageo.z0 + iz);
#pragma unroll
            for (int c = 0; c < 15; ++c) at[c] = __ldg(a.atlas + vx * 15 + c);
            float sum = __fadd_rn(__fadd_rn(__fadd_rn(at[0], at[1]), __fadd_rn(at[2], at[3])),
                                  __fadd_rn(__fadd_rn(at[4], at[5]), __fadd_rn(at[6], at[7])));
#pragma unroll
            for (int k = 8; k < 15; ++k) sum = __fadd_rn(sum, at[k]);
            if (sum == 0.f) at[14] = 1.f;
          } else {
#pragma unroll
            for (int c = 0; c < 15; ++c) at[c] = 0.f;
          }
          if (ncol == 528) { v[12] = at[0]; v[13] = at[1]; v[14] = at[2]; v[15] = at[3]; }
          else {
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = k < 11 ? at[4 + k] : 0.f;
          }
        }
        if (a.out_split) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
          *reinterpret_cast<uint4*>(mine) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(mine + 16) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
          *reinterpret_cast<uint4*>(mine + 32) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(mine + 48) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
          __syncwarp();
          const int boff = (ncol >> 6) * 128 + (ncol & 63);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int half = j >> 1, row = (j & 1) * 16 + (lane >> 1), part = lane & 1;
            const uint4 d = *reinterpret_cast<const uint4*>(stg + row * 80 + half * 32 + part * 16);
            float* crow = reinterpret_cast<float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(myrow), row));
            if (crow) *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(crow) + boff + half * 64 + part * 8) = d;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(mine + 16 * k) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int row = j * 8 + (lane >> 2), part = lane & 3;
            const float4 d = *reinterpret_cast<const float4*>(stg + row * 80 + part * 16);
            if (mw + row < a.M) *reinterpret_cast<float4*>(ctile + (long long)(mw + row) * a.ldc + ncol + part * 4) = d;
          }
        }
        __syncwarp();
      }
      ++ti;
    }
    if (a.dbg && rank == 0 && threadIdx.x == 64) {
      a.dbg[pair * 8 + 5] = (unsigned long long)w_tfull; a.dbg[pair * 8 + 6] = (unsigned long long)(clock64() - tstart);
      a.dbg[pair * 8 + 7] = ti;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();                                     // neither CTA may free TMEM while the pair still uses it
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// plain fp32 [rows][576] -> split bf16 hi|lo blocks (test entry sc_dense_layer only)
__global__ void split_rows_kernel(const float* __restrict__ in, int64_t rows, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * (kFeatLd / 4)) return;
  const int64_t m = i / (kFeatLd / 4);
  const int n = (int)(i - m * (kFeatLd / 4)) * 4;
  const float4 v = __ldg(reinterpret_cast<const float4*>(in + m * kFeatLd + n));
  store_split4(out + m * kFeatLd, n, v.x, v.y, v.z, v.w);
}
int launch_split_rows(sc_ctx* ctx, const float* in, int64_t rows, float* out, cudaStream_t st) {
  const int64_t work = rows * (kFeatLd / 4);
  split_rows_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(in, rows, out);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// row-map mode: which 256-row tiles of the dense slab contain a candidate row at all (one warp per tile)
__global__ void tile_flags_kernel(const int* __restrict__ rowmap, long long num_tiles, int nt, int mt, int Y, int M, long long ldc,
                                  long long c_ys, long long c_zs, unsigned char* __restrict__ flags) {
  const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= num_tiles) return;
  long long r = t / nt;
  const int m_tile = (int)(r % mt); r /= mt;
  const int y = (int)(r % Y);
  const int z = (int)(r / Y);
  const int lane = threadIdx.x & 31;
  bool any = false;
  for (int k = lane; k < 256; k += 32) {
    const int m = m_tile * 256 + k;
    if (m < M && __ldg(rowmap + ((long long)z * c_zs + (long long)y * c_ys + (long long)m * ldc)) >= 0) any = true;
  }
  any = __any_sync(0xffffffffu, any);
  if (lane == 0) flags[t] = any ? 1 : 0;
}

int tc_init(sc_ctx* ctx) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
    cudaGetLastError();
    set_error("tcgen05 back-end: cuTensorMapEncodeTiled unavailable");
    return SC_ERR_UNSUPPORTED;
  }
  TcState* s = new TcState();
  s->encode = reinterpret_cast<EncodeTiledFn>(fn);
  ctx->tc_state = s;
  return SC_OK;
}

void tc_destroy(sc_ctx* ctx) {
  delete reinterpret_cast<TcState*>(ctx->tc_state);
  ctx->tc_state = nullptr;
}

static int pick_bn(int n_store) {
  // widest tile <= 192 (two CTAs x 256 TMEM columns per SM) that wastes the fewest columns
  int best = 16, best_cost = 1 << 30;
  for (int bn = 192; bn >= 32; bn -= 16) {
    const int tiles = (n_store + bn - 1) / bn;
    const int cost = tiles * bn * 4 + tiles * 128;  // padded columns + A re-reads
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

int launch_gemm_tc(sc_ctx* ctx, const GemmProblem& p, const GemmW& w, cudaStream_t st) {
  TcState* s = reinterpret_cast<TcState*>(ctx->tc_state);
  SC_CHECK(s != nullptr, SC_ERR_UNSUPPORTED, "tcgen05 back-end not initialised");
  if (p.M <= 0 || p.Y <= 0 || p.Z <= 0) return SC_OK;
  SC_CHECK(p.kc % TC_BK == 0 && p.ntaps * p.kc == w.Kpad && p.n_store % 4 == 0 && p.n_store <= w.Npad, SC_ERR_ARG,
           "gemm_tc: bad geometry kc=%d ntaps=%d Kpad=%d n_store=%d", p.kc, p.ntaps, w.Kpad, p.n_store);
  TcArgs a;
  a.kpt = p.kc / TC_BK;
  a.c_col0 = p.c_col0;
  a.nkb = p.ntaps * a.kpt;
  a.bn = pick_bn(p.n_store);
  a.out_w = ctx->out_w; a.out_b = ctx->out_b;
  a.atlas = p.atlas; a.ageo = p.ageo;
  a.rowmap = p.rowmap; a.rowvox = p.rowvox; a.crow_ld = 0; a.tile_on = nullptr;
  if (p.sm) {   // fc_2 with the out_layer, softmax and argmax in its epilogue
    SC_CHECK(p.n_store == kH2Ld && p.ntaps == 1 && p.c_col0 == 0 && !p.out_split && !p.rowmap && !p.atlas && w.Npad == kH2Ld,
             SC_ERR_ARG, "gemm_tc: the out_layer epilogue is for fc_2");
    a.sm = *p.sm;
  }
  SC_CHECK(!p.mc_acc || p.sm, SC_ERR_ARG, "gemm_tc: the Monte-Carlo accumulator needs the out_layer epilogue");
  a.mc_acc = p.mc_acc; a.mc_first = p.mc_first;
  a.nt = (p.n_store + a.bn - 1) / a.bn;
  a.mt = (p.M + TC_BM - 1) / TC_BM;
  a.Y = p.Y; a.M = p.M; a.npad = w.Npad;
  a.n_store = (p.n_store + 15) & ~15;     // whole 16-column chunks: the caller lets pad columns be overwritten with zeros
  if (p.atlas) a.n_store = 576;
  SC_CHECK(p.c_col0 % 16 == 0, SC_ERR_ARG, "gemm_tc: c_col0 must be a multiple of 16");
  a.a_y0 = p.a_y0; a.a_z0 = p.a_z0; a.a_swap = p.a_swap;
  for (int t = 0; t < 9; ++t) { a.tap_dx[t] = t < p.ntaps ? p.tap_dx[t] : 0; a.tap_dy[t] = t < p.ntaps ? p.tap_dy[t] : 0; a.tap_dz[t] = t < p.ntaps ? p.tap_dz[t] : 0; }
  a.C = p.C; a.ldc = p.ldc; a.c_ys = p.c_ys; a.c_zs = p.c_zs;
  if (p.rowmap) {   // candidate compaction: the C strides of the dense slab become row counts, rows are kFeatLd floats apart
    SC_CHECK(p.out_split && p.ldc % kFeatLd == 0 && p.c_ys % kFeatLd == 0 && p.c_zs % kFeatLd == 0, SC_ERR_ARG, "gemm_tc: rowmap needs split rows of kFeatLd floats");
    a.crow_ld = kFeatLd; a.ldc = p.ldc / kFeatLd; a.c_ys = p.c_ys / kFeatLd; a.c_zs = p.c_zs / kFeatLd;
  }
  a.bias = w.bias; a.alpha = w.alpha; a.scale = w.scale; a.out_split = p.out_split;
  // CTA pairs (cta_group::2) for the wide streaming-weight tiles, the persistent single-CTA kernel for the narrow ones
  const bool pair = a.bn >= 128 && a.bn % 16 == 0;
  SC_CHECK(!p.rowmap || pair, SC_ERR_ARG, "gemm_tc: the row map is implemented in the CTA-pair kernel");
  SC_CHECK(!p.sm || pair, SC_ERR_ARG, "gemm_tc: the out_layer epilogue is implemented in the CTA-pair kernel");
  SC_CHECK(!p.atlas || (pair && p.c_col0 == 0 && p.n_store == 540 && w.Npad == 576), SC_ERR_ARG, "gemm_tc: the atlas epilogue is for FC1 in the CTA-pair kernel");
  const long long blocks = (long long)a.mt * a.nt * p.Y * p.Z;
  SC_CHECK(blocks < (1ll << 31), SC_ERR_ARG, "gemm_tc: grid too large");
  a.num_tiles = blocks;
  a.dbg = (ctx->tc_timing_cls == p.prof_cls) ? ctx->tc_timing_buf : nullptr;
  a.last_ksteps = 4;
  if (p.ntaps == 1 && w.k_used > w.Kpad - TC_BK && w.k_used <= w.Kpad) a.last_ksteps = (w.k_used - (w.Kpad - TC_BK) + 15) / 16;   // real fan-in inside the last block
  int stage_bytes;
  size_t smem = 0;
  if (pair) {
    a.mt = (p.M + 255) / 256;
    a.num_tiles = (long long)a.mt * a.nt * p.Y * p.Z;
    a.epi_warps = 16;
    stage_bytes = 2 * TC_A_HALF + 2 * (a.bn / 2) * 128;
    SC_CHECK(a.nt <= 4, SC_ERR_ARG, "gemm_tc: more than 4 n-tiles in the CTA-pair kernel");
    const int cst = (a.nt > 2 ? a.nt : 2) * 3 * a.bn * 4;     // resident epilogue constants of every n-tile
    const int budget = 227 * 1024 - 1024 - 192 - 16 - cst - a.epi_warps * 2560;
    a.stages = budget / stage_bytes;
    if (a.stages > 6) a.stages = 6;
    SC_CHECK(a.stages >= 2, SC_ERR_ARG, "gemm_tc: pair tile too wide");
    smem = 1024 + (size_t)a.stages * stage_bytes + (2 * a.stages + 4) * 8 + 32 + cst + (size_t)a.epi_warps * 2560;
  } else {
    a.epi_warps = a.bn > 64 ? 16 : 8;
    const int budget = 227 * 1024 - 1024 - 128 - 16 - 2 * 3 * a.bn * 4 - a.epi_warps * 2560;   // alignment slack, barriers, epilogue constants, store tiles
    stage_bytes = 2 * TC_A_HALF + 2 * a.bn * 128;
    a.stages = budget / stage_bytes;
    if (a.stages > 6) a.stages = 6;
    SC_CHECK(a.stages >= 2, SC_ERR_ARG, "gemm_tc: tile too wide for two stages (bn=%d)", a.bn);
    smem = 1024 + (size_t)a.stages * stage_bytes + (2 * a.stages + 4) * 8 + 16 + 2 * 3 * a.bn * 4 + (size_t)a.epi_warps * 2560;
  }

  CUtensorMap mapA, mapB;
  {
    // a row of kc logical columns is 2*kc bf16 (hi | lo per 64-wide block)
    cuuint64_t dims[4] = {(cuuint64_t)p.a_dims[0] * 2, (cuuint64_t)p.a_dims[1], (cuuint64_t)p.a_dims[2], (cuuint64_t)p.a_dims[3]};
    cuuint64_t strides[3] = {(cuuint64_t)p.a_strides[0] * 4, (cuuint64_t)p.a_strides[1] * 4, (cuuint64_t)p.a_strides[2] * 4};
    cuuint32_t box[4] = {TC_BK, TC_BM, 1, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = s->encode(&mapA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<float*>(p.a_base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "gemm_tc: cuTensorMapEncodeTiled(A) failed with %d (dims %llu %llu %llu %llu)", (int)r,
             (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2], (unsigned long long)dims[3]);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)w.Kpad * 2, (cuuint64_t)w.Npad};
    cuuint64_t strides[1] = {(cuuint64_t)w.Kpad * 4};
    cuuint32_t box[2] = {TC_BK, (cuuint32_t)(pair ? a.bn / 2 : a.bn)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = s->encode(&mapB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.w_nk, dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "gemm_tc: cuTensorMapEncodeTiled(B) failed with %d", (int)r);
  }
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(gemm_tc_persistent_kernel), 227 * 1024));
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(gemm_tc_pair_kernel<false>), 227 * 1024));
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(gemm_tc_pair_kernel<true>), 227 * 1024));
  if (p.mc_acc) SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(gemm_tc_pair_kernel<true, true>), 227 * 1024));
  SC_CHECK(smem <= 227 * 1024, SC_ERR_ARG, "gemm_tc: shared memory budget exceeded (%zu)", smem);
  ProfScope prof(ctx, p.prof_cls, st);
  a.n_mma = a.nt * a.bn;
  if (pair && p.ntaps == 1) {
    // dense layers: the MMAs only produce the real output columns (rounded to 16, at least 32 in the last tile)
    int real = (w.N + 15) & ~15;
    if (real > p.n_store) real = (p.n_store + 15) & ~15;
    if (real - (a.nt - 1) * a.bn >= 32 && real <= a.nt * a.bn) a.n_mma = real;
  }
  if (pair && p.rowmap) {   // skip the tiles of the dense slab without a candidate row
    if (ctx->tile_flags_cap < (size_t)a.num_tiles) {
      if (ctx->tile_flags) cudaFree(ctx->tile_flags);
      ctx->tile_flags = nullptr; ctx->tile_flags_cap = 0;
      const size_t cap = ((size_t)a.num_tiles + 65535) & ~(size_t)65535;
      SC_CUDA(cudaMalloc(&ctx->tile_flags, cap));
      ctx->tile_flags_cap = cap;
    }
    tile_flags_kernel<<<(unsigned)((a.num_tiles + 7) / 8), 256, 0, st>>>(p.rowmap, a.num_tiles, a.nt, a.mt, a.Y, a.M, a.ldc, a.c_ys, a.c_zs, ctx->tile_flags);
    ctx->launches++;
    a.tile_on = ctx->tile_flags;
  }
  if (pair) {
    const long long units = p.sm ? a.num_tiles / a.nt : a.num_tiles;   // work units of the pair kernel (see its tile walk)
    const long long pairs = units < ctx->sm_count / 2 ? units : ctx->sm_count / 2;
    if (p.mc_acc) gemm_tc_pair_kernel<true, true><<<(unsigned)(2 * pairs), 64 + 32 * a.epi_warps, smem, st>>>(mapA, mapB, a);
    else if (p.sm) gemm_tc_pair_kernel<true><<<(unsigned)(2 * pairs), 64 + 32 * a.epi_warps, smem, st>>>(mapA, mapB, a);   // __cluster_dims__(2,1,1)
    else gemm_tc_pair_kernel<false><<<(unsigned)(2 * pairs), 64 + 32 * a.epi_warps, smem, st>>>(mapA, mapB, a);
  } else {
    const unsigned grid = (unsigned)(blocks < ctx->sm_count ? blocks : ctx->sm_count);
    gemm_tc_persistent_kernel<<<grid, 64 + 32 * a.epi_warps, smem, st>>>(mapA, mapB, a);
  }
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
