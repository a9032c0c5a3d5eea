// Strip-sweep implicit-GEMM 3x3 dilated convolution on tcgen05 (sm_100a) for the dense whole-volume path
// (SURVEY.md 8f-1; layers conv2..conv5 of cnn_cort/nets.py:172-177 evaluated at every pixel of a slice).
//
// Map layout ("wide rows"): all slices of a view lie side by side, position (row r, slice s, col c) is pixel
// r * Pw + s * C1 + c with Pw = ns * C1.  A CTA owns a strip of 128 adjacent wide columns and sweeps down the rows:
// every input row of the strip is TMA-loaded ONCE into a shared-memory ring.  With dilation d the rows r, r+d, r+2d
// interact, so a sweep runs over one residue class of rows (r = q + d*n).
//
//   warp 0    TMA producer: one (128 + 2d)-pixel box per input row (two for the 256 B/pixel layout)
//   warp 1    MMA issue, converged, compile-time unrolled: ONE pass per input row.  Class row n feeds output rows
//             n-2, n-1, n through filter rows 2, 1, 0, so the weights stack the three filter rows along N
//             ([W_ky2 | W_ky1 | W_ky0], N = 3*bn) and per (kx, k-step) the bf16x3 split product is three MMAs
//             xh*Wh, xh*Wl, xl*Wh into one D that spans the accumulators of output rows n-2 .. n;
//             column taps are descriptor start offsets inside the row box, weights stay resident (k-step-packed panels)
//   warps 2-17 epilogue (4 lane quarters x 4 column groups): TMEM -> BN scale/shift -> PReLU -> [fused 2x2 stride-1
//             max-pool: horizontal neighbour by shuffle / a small exchange buffer, vertical neighbour = the previous
//             row kept in registers] -> split bf16 hi|lo -> SWIZZLE_128B output tile in shared memory -> one TMA
//             tensor store per row box (no per-thread global addressing; partial boxes are clipped by the TMA unit)
//
// Accumulator ring: S slots of bn TMEM columns plus two spill slots, (S + 2) * bn <= 512.  A per-CTA input-row counter g
// (not reset between items; it starts at 2) numbers the slots: input row g writes slots g-2, g-1, g, i.e. the physical
// columns [p, p + 3) * bn with p = (g - 2) mod S, which never wrap: logical slot l < 2 is physical l + physical S + l.
// An MMA writes its whole D, so no slot can start from zero inside a stacked MMA: every MMA accumulates, and the epilogue
// clears a slot (both parts) after reading it; all slots are cleared once at the start.  Slot g is committed full after
// input row g + 2, always.  An item of nrow output rows reads nrow + 2 input rows: its output rows are its first nrow
// slots, the two before them (the previous item's two halo slots, or two leading slots) hold partial sums that the epilogue
// clears and discards.  Output class row n always lands in slot (n + 2) mod S, so its summation order (one part or two)
// does not depend on how the rows are cut into items or which items are skipped: an item whose first row does not follow
// on from the previous one's slots jumps g ahead by d < S; the previous item's halo slots it does not share are committed
// at once and it claims its own leading slots.  The slot barriers keep their phase parities per slot (bit masks).
//
// Pixel formats: F32CH: 128 B = 32 bf16 hi | 32 bf16 lo (20-channel maps); F64CH: 256 B = 64 hi | 64 lo.
#include "tc_common.cuh"

namespace sc {

constexpr int SW_SLOT_HALF = 17408;   // bytes reserved per TMA box: (128 + 2*4) pixels x 128 B, 1024-aligned
constexpr int SW_MAX_SLOTS = 14;      // accumulator slots (bn = 32); barriers of the largest ring fit SW_BAR_BYTES
constexpr int SW_BAR_BYTES = 512;     // mbarriers + TMEM address slot

struct SweepArgs {
  int Pw, R;              // wide-row pitch (pixels) and number of rows of the map geometry
  int bn;                 // accumulator columns per output row (output channels rounded up to 16)
  int S;                  // accumulator slots of the ring: (S + 2) * bn <= 512 TMEM columns
  int nstrips, strip_w;   // strips start every strip_w wide columns (128, or 128 - pool reach)
  int nseg, L;            // row segments per (strip, class); class rows per segment (output rows of an item)
  int n_items;
  int stages;
  int out_bufs;           // output tiles in shared memory (2: double-buffered, 1 when shared memory is short)
  int npanels;            // weight panels (4 k-steps each)
  int in_dx, in_dy;       // offset (pixels, rows) of the input window against the output position: 0 for a valid convolution,
                          // -2 for the full correlation of a dgrad (what lies outside the map is zero-filled by the TMA unit)
  const float* scale; const float* shift; const float* alpha;
  unsigned long long* dbg;   // optional per-CTA cycle counters [8] (sc_set_option "tc_timing"): where each role waits
  const uint8_t* item_on;    // sparse candidate masks: item t is computed only if item_on[t] != 0 (nullptr: every item)
  double* stats;             // training forward (DIL = 1, no pool): per-channel sum / sum of squares of the raw output over the valid
  int st_H, st_pitch;        // region (row < st_H, (wide column mod st_pitch) < st_H; st_pitch a power of two) accumulated into stats[c][2]
};

__device__ __forceinline__ void sweep_mma(uint32_t acc, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate, uint32_t elected) {
  // descriptors: low word = (addr >> 4) | version/LBO bits, high word constant (SBO 1024 B, SWIZZLE_128B)
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "mov.b64 da, {%1, %6};\n\t"
      "mov.b64 db, {%2, %6};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "}" ::"r"(acc), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(elected), "r"(0x40004040u) : "memory");
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
// BatchNorm batch statistics fused into the training forward sweeps: every epilogue thread keeps the sums of its pixel column,
// folded at the end of the kernel: warp shuffles -> shared memory across the four lane quarters -> one double atomic per CTA,
// channel and moment (the per-CTA global atomics hit the same few addresses: ~ 27 clk each, so there must be few of them)
template <int CW>
__device__ __forceinline__ void sweep_stats_flush(float (&st_s)[CW], float (&st_q)[CW], float* s_red /*[16 warps][2 * CW]*/, int ew, int c0,
                                                  bool real, int lane, double* stats) {
#pragma unroll
  for (int k = 0; k < CW; ++k)
#pragma unroll
    for (int o = 16; o; o >>= 1) { st_s[k] += __shfl_xor_sync(0xffffffffu, st_s[k], o); st_q[k] += __shfl_xor_sync(0xffffffffu, st_q[k], o); }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < CW; ++k) { s_red[ew * 2 * CW + k] = st_s[k]; s_red[ew * 2 * CW + CW + k] = st_q[k]; }
  }
  asm volatile("bar.sync 7, 512;" ::: "memory");      // its own barrier: 5 and 6 belong to the row loop, which slower warps may still be in
  if ((ew & 3) == 0 && real && lane < 2 * CW) {  // first warp of every column group: lane -> (moment, channel)
    const int base = ew * 2 * CW + lane;         // the group's four warps (one per TMEM lane quarter) are ew, ew + 1, ew + 2, ew + 3
    const float tot = s_red[base] + s_red[base + 2 * CW] + s_red[base + 4 * CW] + s_red[base + 6 * CW];
    const int mom = lane / CW, ch = c0 + (lane - mom * CW);
    if (ch < 64) atomicAdd(&stats[ch * 2 + mom], (double)tot);
  }
}

template <int CW>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&r)[CW]) {
  if constexpr (CW == 16) tmem_ld16(taddr, r); else tmem_ld8(taddr, r);
}
template <int CW>
__device__ __forceinline__ void tmem_zero(uint32_t taddr) {
  if constexpr (CW == 16)
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
                 ::"r"(taddr), "r"(0u) : "memory");
  else
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(0u) : "memory");
}
// every accumulator column of this warp's lanes and column group starts at zero (the MMAs only ever accumulate)
template <int CW>
__device__ __forceinline__ void sweep_acc_clear(uint32_t tcol, int S, int bn) {
  for (int j = 0; j < S + 2; ++j) tmem_zero<CW>(tcol + (uint32_t)(j * bn));
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// Epilogue side of the accumulator ring: wait for slot dj (phase parities: bit mask dph), read it into acc if `keep` (summing the
// spill part of slots 0 and 1), clear it, hand it back to the MMA warp (aempty, of the leader CTA for PAIR), advance to the next slot.
// tcol = TMEM address of this warp's lane quarter and first column; `real` = the warp's columns are computed ones.
template <int CW, bool PAIR>
__device__ __forceinline__ void sweep_drain(uint64_t* afull, uint64_t* aempty, uint32_t& dj, uint32_t& dph, int S, int bn,
                                            uint32_t tcol, bool real, bool keep, int lane, float (&acc)[CW], bool timed,
                                            uint32_t& w_wait) {
  const long long c0 = timed ? clock64() : 0;
  mbar_wait(&afull[dj], (dph >> dj) & 1u);
  dph ^= 1u << dj;
  if (timed) w_wait += (uint32_t)(clock64() - c0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (real) {
    const uint32_t taddr = tcol + dj * (uint32_t)bn, tspill = taddr + (uint32_t)(S * bn);
    const bool split = dj < 2;               // warp-uniform
    if (keep) {
#pragma unroll
      for (int h = 0; h < CW; h += 8) {      // 8 columns at a time: the spill part costs no extra registers
        uint32_t r1[8], r2[8];
        tmem_ld8(taddr + h, r1);
        if (split) tmem_ld8(tspill + h, r2);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[h + k] = split ? __uint_as_float(r1[k]) + __uint_as_float(r2[k]) : __uint_as_float(r1[k]);
      }
    }
    tmem_zero<CW>(taddr);
    if (split) tmem_zero<CW>(tspill);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncwarp();
  if (lane == 0) {
    if (PAIR) mbar_arrive_cta(&aempty[dj], 0); else mbar_arrive(&aempty[dj]);
  }
  if (++dj == (uint32_t)S) dj = 0;
}
// MMA side: wait until slot j's previous use has been drained (phase parities: bit mask eph)
__device__ __forceinline__ void sweep_claim(uint64_t* aempty, uint32_t j, uint32_t& eph) {
  mbar_wait(&aempty[j], ((eph >> j) & 1u) ^ 1u);
  eph ^= 1u << j;
}
__device__ __forceinline__ uint32_t slot_back(uint32_t j, uint32_t k, int S) { return j >= k ? j - k : j + (uint32_t)S - k; }   // k <= 2
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// KSTEPS: 16-channel k-steps per tap; DIL: dilation; POOL: 1 = fuse the stride-1 max-pool with window {0, DIL}^2 (dense maps),
// 2 = fuse the 2x2 stride-2 max-pool (patch maps: output pitch and rows halve, row segments start on even rows);
// CW: accumulator columns per epilogue warp (8 or 16; 4 column groups); LO64: lo operand 64 B into the row (F32CH)
// instead of in its own box; OUT32: output pixels are F32CH
template <int KSTEPS, int DIL, int POOL, int CW, bool LO64, bool OUT32>
__global__ void __launch_bounds__(576, 1)
conv_sweep_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapO,
                  const SweepArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int BOXPX = 128 + 2 * DIL;
  constexpr int BOX_BYTES = BOXPX * 128;
  constexpr int NBOX = LO64 ? 1 : 2;
  constexpr int SLOT = NBOX * SW_SLOT_HALF;
  constexpr int LO_OFF = LO64 ? 64 : SW_SLOT_HALF;
  const int half_bytes = 3 * a.bn * 128;                               // W hi (or lo) rows of one panel, stacked filter rows
  const int panel_bytes = 2 * half_bytes;
  const int w_bytes = a.npanels * panel_bytes;
  uint8_t* sW = smem;
  uint8_t* sRing = smem + w_bytes;
  constexpr int OB_BYTES = OUT32 ? 16384 : 32768;                      // one output row tile: 128 pixels, hi box [+ lo box]
  uint8_t* sOut = sRing + a.stages * SLOT;                             // 1024-aligned (SLOT, w_bytes are multiples of 1024)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + a.out_bufs * OB_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + a.stages;
  uint64_t* afull = bars + 2 * a.stages;   // [S] accumulator slot complete (MMA commit)
  uint64_t* aempty = afull + a.S;          // [S] accumulator slot read and cleared (16 epilogue warps)
  uint64_t* wfull = aempty + a.S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wfull + 1);
  float* s_const = reinterpret_cast<float*>(tmem_slot + 2);            // [scale 64 | shift 64 | alpha 64]
  float* s_xch = s_const + 192;                                        // [2 row parities][4 groups][4 quarters][2][16]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int j = 0; j < a.S; ++j) { mbar_init(&afull[j], 1); mbar_init(&aempty[j], 16); }
    mbar_init(wfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = threadIdx.x; i < 64; i += blockDim.x) {
    const bool ok = i < a.bn;
    s_const[i] = ok ? __ldg(a.scale + i) : 0.f;
    s_const[64 + i] = ok ? __ldg(a.shift + i) : 0.f;
    s_const[128 + i] = ok ? __ldg(a.alpha + i) : 0.f;
  }
  for (int i = threadIdx.x; i < a.out_bufs * OB_BYTES / 16; i += blockDim.x)   // channel padding of the output tiles stays zero
    reinterpret_cast<uint4*>(sOut)[i] = make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  // epilogue geometry: TMEM lane quarter, column group and the first accumulator column of this warp
  const int q4 = warp & 3, ew = warp - 2, grp = ew >> 2, c0 = grp * CW;
  const bool real = c0 < a.bn;             // groups beyond the computed columns only take part in the barriers
  const uint32_t tcol = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)c0;
  if (warp >= 2 && real) sweep_acc_clear<CW>(tcol, a.S, a.bn);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  // item -> (strip, class q, segment); identical in every role
  auto decode = [&](int item, int& w0, int& q, int& n0, int& Lc) {
    const int strip = item % a.nstrips;
    const int rest = item / a.nstrips;
    q = rest % DIL;
    const int seg = rest / DIL;
    w0 = strip * a.strip_w;
    const int Nq = (a.R - q + DIL - 1) / DIL;      // class rows
    n0 = seg * a.L;
    Lc = Nq - n0 < a.L ? Nq - n0 : a.L;            // output class rows of this item (may be <= 0: nothing to do)
  };

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapW)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapO)) : "memory");
      mbar_expect_tx(wfull, (uint32_t)w_bytes);
      for (int p = 0; p < 2 * a.npanels; ++p) tma_load_2d(&mapW, wfull, sW + p * half_bytes, 0, p * 3 * a.bn);
      uint32_t g = 0;
      long long w_empty = 0;
      const long long tstart = a.dbg ? clock64() : 0;
      for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        int w0, q, n0, Lc;
        decode(item, w0, q, n0, Lc);
        if (Lc <= 0 || (a.item_on && !a.item_on[item])) continue;
        const int nload = Lc + (POOL == 1 ? 1 : 0) + 2;
        for (int m = 0; m < nload; ++m, ++g) {
          const uint32_t s = g % a.stages, use = g / a.stages;
          if (use > 0) {
            const long long c0 = a.dbg ? clock64() : 0;
            mbar_wait(&empty[s], (use - 1) & 1);
            if (a.dbg) w_empty += clock64() - c0;
          }
          mbar_expect_tx(&full[s], (uint32_t)(NBOX * BOX_BYTES));
          uint8_t* sp = sRing + s * SLOT;
          const int r = q + DIL * (n0 + m);          // rows beyond the map are zero-filled by the TMA unit
          tma_load_3d(&mapA, &full[s], sp, 0, w0 + a.in_dx, r + a.in_dy);
          if (NBOX == 2) tma_load_3d(&mapA, &full[s], sp + SW_SLOT_HALF, 64, w0 + a.in_dx, r + a.in_dy);
        }
      }
      if (a.dbg) { a.dbg[blockIdx.x * 8 + 0] = (unsigned long long)w_empty; a.dbg[blockIdx.x * 8 + 1] = (unsigned long long)(clock64() - tstart); }
    }
    __syncwarp();
  } else if (warp == 1) {
    const uint32_t leader = elect_one();
    // D = F32, A = B = BF16, K-major, N = 3 * bn (stacked filter rows), M = 128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(3 * a.bn >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    mbar_wait(wfull, 0);
    const uint32_t w_lo = desc_lo(smem_u32(sW));
    const uint32_t ring_lo = desc_lo(smem_u32(sRing));
    const uint32_t panel16 = (uint32_t)(panel_bytes >> 4), wl_off = (uint32_t)(half_bytes >> 4);
    uint32_t rs = 0, rph = 0;                  // ring stage / phase parity of the next input row
    uint32_t j = 2, eph = 0;                   // its accumulator slot g mod S (g starts at 2), slot phase parities
    bool open = false;                         // the last computed item's halo slots await their commit
    long long w_full = 0, w_tempty = 0;
    const long long tstart = a.dbg ? clock64() : 0;
    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
      int w0, q, n0, Lc;
      decode(item, w0, q, n0, Lc);
      if (Lc <= 0 || (a.item_on && !a.item_on[item])) continue;
      const int nin = Lc + (POOL == 1 ? 1 : 0) + 2;
      const uint32_t j0 = (uint32_t)(n0 + 2) % (uint32_t)a.S;     // slot of the item's first output row
      const uint32_t d = open ? (j0 + (uint32_t)a.S - j) % (uint32_t)a.S : 2u;
      if (d) {                                 // not following on: flush the unshared old halo slots, claim the new leading ones
        if (open && leader) { umma_commit(&afull[slot_back(j, 2, a.S)]); if (d >= 2) umma_commit(&afull[slot_back(j, 1, a.S)]); }
        if (d >= 2) sweep_claim(aempty, slot_back(j0, 2, a.S), eph);
        sweep_claim(aempty, slot_back(j0, 1, a.S), eph);
      }
      j = j0; open = true;
      for (int m = 0; m < nin; ++m) {
        long long c0 = a.dbg ? clock64() : 0;
        sweep_claim(aempty, j, eph);             // slot g: its previous use has been read and cleared
        if (a.dbg) { const long long c1 = clock64(); w_tempty += c1 - c0; c0 = c1; }
        mbar_wait(&full[rs], rph);
        if (a.dbg) w_full += clock64() - c0;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t p = slot_back(j, 2, a.S);                    // slots g-2 .. g = physical slots p .. p+2
        const uint32_t acc = tmem_base + p * (uint32_t)a.bn;
        const uint32_t sl = ring_lo + rs * (SLOT >> 4);
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            const int gk = kx * KSTEPS + ks;                            // compile-time after unrolling
            const uint32_t a_hi = sl + (uint32_t)(kx * DIL * 8 + ks * 2);
            const uint32_t a_lo = a_hi + (uint32_t)(LO_OFF >> 4);
            const uint32_t wh = w_lo + (uint32_t)(gk >> 2) * panel16 + (uint32_t)((gk & 3) * 2);
            sweep_mma(acc, a_lo, wh, idesc, 1, leader);
            sweep_mma(acc, a_hi, wh + wl_off, idesc, 1, leader);
            sweep_mma(acc, a_hi, wh, idesc, 1, leader);
          }
        }
        if (leader) {
          umma_commit(&empty[rs]);
          umma_commit(&afull[p]);                // slot g-2 has all three filter rows
        }
        __syncwarp();
        if (++rs == (uint32_t)a.stages) { rs = 0; rph ^= 1; }
        if (++j == (uint32_t)a.S) j = 0;
      }
    }
    if (open && leader) {                        // the CTA's last two slots (halo rows) get no later input row
      umma_commit(&afull[slot_back(j, 2, a.S)]);
      umma_commit(&afull[slot_back(j, 1, a.S)]);
    }
    __syncwarp();
    if (a.dbg && leader) {
      a.dbg[blockIdx.x * 8 + 2] = (unsigned long long)w_full; a.dbg[blockIdx.x * 8 + 3] = (unsigned long long)w_tempty;
      a.dbg[blockIdx.x * 8 + 4] = (unsigned long long)(clock64() - tstart);
    }
  } else {
    const int px = q4 * 32 + lane;           // pixel inside the strip = row of the output tile
    const bool issuer = threadIdx.x == 64;
    // byte offsets of this thread's hi / lo pieces inside a tile (SWIZZLE_128B: 16 B chunk index ^= row & 7)
    const int trow = POOL == 2 ? px >> 1 : px; // row of the output tile this thread writes (stride-2 pool: even lanes only)
    const bool writer = POOL == 2 ? !(lane & 1) : true;
    const uint32_t row_off = (uint32_t)trow * 128u;
    const uint32_t sw = (uint32_t)(trow & 7);
    const uint32_t hi_chunk = (uint32_t)(c0 >> 3);
    const uint32_t lo_base = OUT32 ? 0u : 16384u, lo_chunk = OUT32 ? 4u + hi_chunk : hi_chunk;
    uint32_t t = 0, e = 0;                   // conv rows consumed, rows emitted
    uint32_t dj = 0, dph = 0;                // accumulator slot to drain next, slot phase parities
    uint32_t w_tfull = 0;
    const bool timed = a.dbg != nullptr;
    const long long tstart = a.dbg ? clock64() : 0;
    constexpr bool STATS = POOL == 0 && DIL == 1;   // the instantiations the training forward uses
    float st_s[STATS ? CW : 1], st_q[STATS ? CW : 1];
#pragma unroll
    for (int k = 0; k < (STATS ? CW : 1); ++k) st_s[k] = st_q[k] = 0.f;
    float v[CW];
    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
      int w0, q, n0, Lc;
      decode(item, w0, q, n0, Lc);
      if (Lc <= 0 || (a.item_on && !a.item_on[item])) continue;
      const int nrow = Lc + (POOL == 1 ? 1 : 0);
      // halo slots of the previous item (dj = its first one) up to the new item's two leading ones, as the MMA warp jumps
      const uint32_t j0 = (uint32_t)(n0 + 2) % (uint32_t)a.S;
      const uint32_t d = (j0 + 2u * (uint32_t)a.S - 2u - dj) % (uint32_t)a.S;
      if (t == 0 || d >= 3) {
        if (t > 0)
          for (int h = 0; h < 2; ++h) sweep_drain<CW, false>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
        dj = slot_back(j0, 2, a.S);
      } else {
        for (uint32_t h = 0; h < d; ++h) sweep_drain<CW, false>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
      }
      for (int h = 0; h < 2; ++h) sweep_drain<CW, false>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
      float hprev[CW];
#pragma unroll
      for (int k = 0; k < CW; ++k) hprev[k] = 0.f;
      for (int m = 0; m < nrow; ++m, ++t) {
        sweep_drain<CW, false>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, true, lane, v, timed, w_tfull);
        if (real) {
#pragma unroll
          for (int k4 = 0; k4 < CW / 4; ++k4) {
            const float4 sc_ = *reinterpret_cast<const float4*>(s_const + c0 + 4 * k4);
            const float4 sh = *reinterpret_cast<const float4*>(s_const + 64 + c0 + 4 * k4);
            const float4 al = *reinterpret_cast<const float4*>(s_const + 128 + c0 + 4 * k4);
            v[4 * k4 + 0] = prelu(fmaf(v[4 * k4 + 0], sc_.x, sh.x), al.x);
            v[4 * k4 + 1] = prelu(fmaf(v[4 * k4 + 1], sc_.y, sh.y), al.y);
            v[4 * k4 + 2] = prelu(fmaf(v[4 * k4 + 2], sc_.z, sh.z), al.z);
            v[4 * k4 + 3] = prelu(fmaf(v[4 * k4 + 3], sc_.w, sh.w), al.w);
          }
        }

        int r_out = q + DIL * (n0 + m);
        if (POOL == 1) {
          // horizontal neighbour (DIL pixels to the right): same warp by shuffle, next quarter through shared memory
          if (real) {
            float* xw = s_xch + (((t & 1) * 4 + grp) * 4 + q4) * 32;      // [row parity][group][quarter][pd][16]
            if (lane < DIL) {
#pragma unroll
              for (int k4 = 0; k4 < CW / 4; ++k4)
                *reinterpret_cast<float4*>(xw + lane * 16 + 4 * k4) = make_float4(v[4 * k4], v[4 * k4 + 1], v[4 * k4 + 2], v[4 * k4 + 3]);
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
            const bool edge = lane >= 32 - DIL;
            const float* xr = s_xch + (((t & 1) * 4 + grp) * 4 + ((q4 + 1) & 3)) * 32 + (edge ? (lane - (32 - DIL)) * 16 : 0);
#pragma unroll
            for (int k4 = 0; k4 < CW / 4; ++k4) {
              const float4 x4 = *reinterpret_cast<const float4*>(xr + 4 * k4);
              const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float nb = __shfl_down_sync(0xffffffffu, v[4 * k4 + k], DIL);
                if (edge) nb = xs[k];
                const float h = fmaxf(v[4 * k4 + k], nb);
                v[4 * k4 + k] = fmaxf(h, hprev[4 * k4 + k]);     // vertical neighbour: previous class row
                hprev[4 * k4 + k] = h;
              }
            }
          }
          if (m == 0) continue;                    // block-uniform: the first conv row of an item only primes the pool
          r_out -= DIL;
        }
        if (POOL == 2) {
          // 2x2 stride-2 max-pool: pixel pairs (2j, 2j+1) never straddle a lane quarter, row pairs (2k, 2k+1) lie inside
          // an item (segments start on even rows); even lanes hold the pooled pixel j = px / 2 after an odd row
          if (real) {
#pragma unroll
            for (int k = 0; k < CW; ++k) {
              const float h = fmaxf(v[k], __shfl_down_sync(0xffffffffu, v[k], 1));
              v[k] = fmaxf(h, hprev[k]);
              hprev[k] = (m & 1) ? 0.f : h;
            }
          }
          if (!(m & 1)) continue;                  // block-uniform
          r_out >>= 1;
        }
        if constexpr (STATS) {
          if (a.stats && real) {
            const int wpx = w0 + px;
            if (wpx < a.Pw && (wpx & (a.st_pitch - 1)) < a.st_H && r_out < a.st_H) {
#pragma unroll
              for (int k = 0; k < CW; ++k) { st_s[k] += v[k]; st_q[k] = fmaf(v[k], v[k], st_q[k]); }
            }
          }
        }
        // ---- emit row r_out: pieces -> swizzled output tile -> TMA store
        uint8_t* ob = sOut + (e % (uint32_t)a.out_bufs) * OB_BYTES;
        if (a.out_bufs == 1) {                      // single tile: wait until the previous store has read it
          if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync 5, 512;" ::: "memory");
        }
        if (real) {
          uint32_t hi[CW / 2], lo[CW / 2];
#pragma unroll
          for (int k = 0; k < CW / 2; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
#pragma unroll
          for (int c = 0; c < CW / 8; ++c) {
            if (!writer) break;
            *reinterpret_cast<uint4*>(ob + row_off + (((hi_chunk + c) ^ sw) << 4)) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
            *reinterpret_cast<uint4*>(ob + lo_base + row_off + (((lo_chunk + c) ^ sw) << 4)) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        if (a.out_bufs == 2 && issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the other tile is free again
        asm volatile("bar.sync 6, 512;" ::: "memory");
        if (issuer) {
          tma_store_3d(&mapO, ob, 0, POOL == 2 ? w0 >> 1 : w0, r_out);
          if (!OUT32) tma_store_3d(&mapO, ob + 16384, 64, POOL == 2 ? w0 >> 1 : w0, r_out);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        ++e;
      }
    }
    if (t > 0)                               // the last item's two halo slots
      for (int h = 0; h < 2; ++h) sweep_drain<CW, false>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if constexpr (STATS) {
      if (a.stats) sweep_stats_flush<CW>(st_s, st_q, s_xch, ew, c0, real, lane, a.stats);
    }
    if (a.dbg && threadIdx.x == 64) {
      a.dbg[blockIdx.x * 8 + 5] = (unsigned long long)w_tfull; a.dbg[blockIdx.x * 8 + 6] = (unsigned long long)(clock64() - tstart);
      a.dbg[blockIdx.x * 8 + 7] = t;
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
// CTA-pair variant (cta_group::2) for the 40-channel-input layers (conv4 + pool2, conv5), whose resident weights do
// not leave room for a ring in one CTA.  A cluster of two CTAs sweeps two adjacent strips in lock-step:
//   * every CTA loads its own strip's rows, but only HALF of the stacked weight rows (N split across the pair)
//   * both producers signal the LEADER's full barrier; the leader's MMA warp issues tcgen05.mma.cta_group::2 (M = 256)
//     in the stacked order of conv_sweep_kernel (D's first 1.5 bn columns take the leader's weight rows, the rest the
//     peer's) and multicasts its commits to both CTAs
//   * every CTA's epilogue drains its own 128 TMEM lanes and arrives remotely on the leader's accumulator-empty barriers
// Input and output pixels are 256 B (64 hi | 64 lo); 4 column groups of 16.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sweep_mma_2sm(uint32_t acc, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate, uint32_t elected) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "mov.b64 da, {%1, %6};\n\t"
      "mov.b64 db, {%2, %6};\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t"
      "}" ::"r"(acc), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(elected), "r"(0x40004040u) : "memory");
}

template <int KSTEPS, int DIL, int POOL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(576, 1)
conv_sweep_pair_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapO,
                       const SweepArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int BOXPX = 128 + 2 * DIL;
  constexpr int BOX_BYTES = BOXPX * 128;
  constexpr int SLOT = 2 * SW_SLOT_HALF;
  constexpr int CW = 16;
  const int panel_bytes = 3 * a.bn * 128;                               // this CTA's half: 1.5 bn stacked rows of W hi, then of W lo
  const int w_bytes = a.npanels * panel_bytes;
  uint8_t* sW = smem;
  uint8_t* sRing = smem + ((w_bytes + 1023) & ~1023);
  constexpr int OB_BYTES = 32768;
  uint8_t* sOut = sRing + a.stages * SLOT;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + a.out_bufs * OB_BYTES);
  uint64_t* full = bars;                        // leader only: both producers signal it
  uint64_t* empty = bars + a.stages;            // per CTA, arrived by the leader's multicast commit
  uint64_t* afull = bars + 2 * a.stages;        // [S] per CTA, arrived by the leader's multicast commit
  uint64_t* aempty = afull + a.S;               // [S] leader only: both CTAs' epilogue warps arrive
  uint64_t* wfull = aempty + a.S;               // leader only: both CTAs' weight halves
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wfull + 1);
  float* s_const = reinterpret_cast<float*>(tmem_slot + 2);
  float* s_xch = s_const + 192;                 // pooled layers only

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int j = 0; j < a.S; ++j) { mbar_init(&afull[j], 1); mbar_init(&aempty[j], 32); }
    mbar_init(wfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int i = threadIdx.x; i < 64; i += blockDim.x) {
    const bool ok = i < a.bn;
    s_const[i] = ok ? __ldg(a.scale + i) : 0.f;
    s_const[64 + i] = ok ? __ldg(a.shift + i) : 0.f;
    s_const[128 + i] = ok ? __ldg(a.alpha + i) : 0.f;
  }
  for (int i = threadIdx.x; i < a.out_bufs * OB_BYTES / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(sOut)[i] = make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const int q4 = warp & 3, ew = warp - 2, grp = ew >> 2, c0 = grp * CW;
  const bool real = c0 < a.bn;
  const uint32_t tcol = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)c0;
  if (warp >= 2 && real) sweep_acc_clear<CW>(tcol, a.S, a.bn);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();                           // the leader's first MMAs write both CTAs' cleared accumulators
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  // pair item -> (strip pair, class q, segment); this CTA's strip is 2 * strip_pair + rank
  const int nsp = (a.nstrips + 1) >> 1;
  auto decode = [&](int item, int& w0, int& q, int& n0, int& Lc) {
    const int sp = item % nsp;
    const int rest = item / nsp;
    q = rest % DIL;
    const int seg = rest / DIL;
    w0 = (2 * sp + (int)rank) * a.strip_w;       // may lie beyond the map: loads are zero-filled, stores clipped
    const int Nq = (a.R - q + DIL - 1) / DIL;
    n0 = seg * a.L;
    Lc = Nq - n0 < a.L ? Nq - n0 : a.L;
  };

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapW)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapO)) : "memory");
      {
        const uint32_t lbar = smem_u32(wfull) & 0xFEFFFFFFu;            // the leader's barrier (peer bit cleared)
        if (rank == 0) mbar_expect_tx(wfull, (uint32_t)(2 * w_bytes));
        for (int p = 0; p < a.npanels; ++p) tma_load_2d_2sm(&mapW, lbar, sW + p * panel_bytes, 0, (p * 2 + (int)rank) * 3 * a.bn);
      }
      uint32_t g = 0;
      long long w_empty = 0;
      const long long tstart = a.dbg ? clock64() : 0;
      for (int item = pair; item < a.n_items; item += npairs) {
        int w0, q, n0, Lc;
        decode(item, w0, q, n0, Lc);
        if (Lc <= 0 || (a.item_on && !a.item_on[item])) continue;
        const int nload = Lc + (POOL == 1 ? 1 : 0) + 2;
        for (int m = 0; m < nload; ++m, ++g) {
          const uint32_t s = g % a.stages, use = g / a.stages;
          if (use > 0) {
            const long long c0w = a.dbg ? clock64() : 0;
            mbar_wait(&empty[s], (use - 1) & 1);
            if (a.dbg) w_empty += clock64() - c0w;
          }
          const uint32_t lbar = smem_u32(&full[s]) & 0xFEFFFFFFu;
          if (rank == 0) mbar_expect_tx(&full[s], (uint32_t)(2 * 2 * BOX_BYTES));   // both CTAs' boxes land on it
          uint8_t* sp = sRing + s * SLOT;
          const int r = q + DIL * (n0 + m);
          tma_load_3d_2sm(&mapA, lbar, sp, 0, w0 + a.in_dx, r + a.in_dy);
          tma_load_3d_2sm(&mapA, lbar, sp + SW_SLOT_HALF, 64, w0 + a.in_dx, r + a.in_dy);
        }
      }
      if (a.dbg) { a.dbg[blockIdx.x * 8 + 0] = (unsigned long long)w_empty; a.dbg[blockIdx.x * 8 + 1] = (unsigned long long)(clock64() - tstart); }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (rank == 0) {
      const uint32_t leader = elect_one();
      // D = F32, A = B = BF16, K-major, N = 3 * bn (1.5 bn stacked weight rows from each CTA), M = 256
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(3 * a.bn >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      mbar_wait(wfull, 0);
      const uint32_t w_lo = desc_lo(smem_u32(sW));
      const uint32_t ring_lo = desc_lo(smem_u32(sRing));
      const uint32_t panel16 = (uint32_t)(panel_bytes >> 4);
      const uint32_t wl_off = (uint32_t)(3 * a.bn / 2 * 128) >> 4;   // W lo rows follow the 1.5 bn W hi rows
      uint32_t rs = 0, rph = 0, j = 2, eph = 0;                      // as in conv_sweep_kernel
      bool open = false;
      long long w_full = 0, w_tempty = 0;
      const long long tstart = a.dbg ? clock64() : 0;
      for (int item = pair; item < a.n_items; item += npairs) {
        int w0, q, n0, Lc;
        decode(item, w0, q, n0, Lc);
        if (Lc <= 0 || (a.item_on && !a.item_on[item])) continue;
        const int nin = Lc + (POOL == 1 ? 1 : 0) + 2;
        const uint32_t j0 = (uint32_t)(n0 + 2) % (uint32_t)a.S;
        const uint32_t d = open ? (j0 + (uint32_t)a.S - j) % (uint32_t)a.S : 2u;
        if (d) {
          if (open && leader) { umma_commit_2sm(&afull[slot_back(j, 2, a.S)]); if (d >= 2) umma_commit_2sm(&afull[slot_back(j, 1, a.S)]); }
          if (d >= 2) sweep_claim(aempty, slot_back(j0, 2, a.S), eph);
          sweep_claim(aempty, slot_back(j0, 1, a.S), eph);
        }
        j = j0; open = true;
        for (int m = 0; m < nin; ++m) {
          long long c0w = a.dbg ? clock64() : 0;
          sweep_claim(aempty, j, eph);
          if (a.dbg) { const long long c1 = clock64(); w_tempty += c1 - c0w; c0w = c1; }
          mbar_wait(&full[rs], rph);
          if (a.dbg) w_full += clock64() - c0w;
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t p = slot_back(j, 2, a.S);
          const uint32_t acc = tmem_base + p * (uint32_t)a.bn;
          const uint32_t sl = ring_lo + rs * (SLOT >> 4);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
            for (int ks = 0; ks < KSTEPS; ++ks) {
              const int gk = kx * KSTEPS + ks;
              const uint32_t a_hi = sl + (uint32_t)(kx * DIL * 8 + ks * 2);
              const uint32_t a_lo = a_hi + (uint32_t)(SW_SLOT_HALF >> 4);
              const uint32_t wh = w_lo + (uint32_t)(gk >> 2) * panel16 + (uint32_t)((gk & 3) * 2);
              sweep_mma_2sm(acc, a_lo, wh, idesc, 1, leader);
              sweep_mma_2sm(acc, a_hi, wh + wl_off, idesc, 1, leader);
              sweep_mma_2sm(acc, a_hi, wh, idesc, 1, leader);
            }
          }
          if (leader) {
            umma_commit_2sm(&empty[rs]);
            umma_commit_2sm(&afull[p]);
          }
          __syncwarp();
          if (++rs == (uint32_t)a.stages) { rs = 0; rph ^= 1; }
          if (++j == (uint32_t)a.S) j = 0;
        }
      }
      if (open && leader) {
        umma_commit_2sm(&afull[slot_back(j, 2, a.S)]);
        umma_commit_2sm(&afull[slot_back(j, 1, a.S)]);
      }
      __syncwarp();
      if (a.dbg && leader) {
        a.dbg[blockIdx.x * 8 + 2] = (unsigned long long)w_full; a.dbg[blockIdx.x * 8 + 3] = (unsigned long long)w_tempty;
        a.dbg[blockIdx.x * 8 + 4] = (unsigned long long)(clock64() - tstart);
      }
    }
  } else {
    const int px = q4 * 32 + lane;
    const bool issuer = threadIdx.x == 64;
    const int trow = POOL == 2 ? px >> 1 : px;
    const bool writer = POOL == 2 ? !(lane & 1) : true;
    const uint32_t row_off = (uint32_t)trow * 128u;
    const uint32_t sw = (uint32_t)(trow & 7);
    const uint32_t hi_chunk = (uint32_t)(c0 >> 3);
    uint32_t t = 0, e = 0, dj = 0, dph = 0;
    uint32_t w_tfull = 0;
    const bool timed = a.dbg != nullptr;
    const long long tstart = a.dbg ? clock64() : 0;
    constexpr bool STATS = POOL == 0 && DIL == 1;
    float st_s[STATS ? CW : 1], st_q[STATS ? CW : 1];
#pragma unroll
    for (int k = 0; k < (STATS ? CW : 1); ++k) st_s[k] = st_q[k] = 0.f;
    float v[CW];
    for (int item = pair; item < a.n_items; item += npairs) {
      int w0, q, n0, Lc;
      decode(item, w0, q, n0, Lc);
      if (Lc <= 0 || (a.item_on && !a.item_on[item])) continue;
      const int nrow = Lc + (POOL == 1 ? 1 : 0);
      // halo slots of the previous item (dj = its first one) up to the new item's two leading ones, as the MMA warp jumps
      const uint32_t j0 = (uint32_t)(n0 + 2) % (uint32_t)a.S;
      const uint32_t d = (j0 + 2u * (uint32_t)a.S - 2u - dj) % (uint32_t)a.S;
      if (t == 0 || d >= 3) {
        if (t > 0)
          for (int h = 0; h < 2; ++h) sweep_drain<CW, true>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
        dj = slot_back(j0, 2, a.S);
      } else {
        for (uint32_t h = 0; h < d; ++h) sweep_drain<CW, true>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
      }
      for (int h = 0; h < 2; ++h) sweep_drain<CW, true>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
      float hprev[CW];
#pragma unroll
      for (int k = 0; k < CW; ++k) hprev[k] = 0.f;
      for (int m = 0; m < nrow; ++m, ++t) {
        sweep_drain<CW, true>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, true, lane, v, timed, w_tfull);
        if (real) {
#pragma unroll
          for (int k4 = 0; k4 < CW / 4; ++k4) {
            const float4 sc_ = *reinterpret_cast<const float4*>(s_const + c0 + 4 * k4);
            const float4 sh = *reinterpret_cast<const float4*>(s_const + 64 + c0 + 4 * k4);
            const float4 al = *reinterpret_cast<const float4*>(s_const + 128 + c0 + 4 * k4);
            v[4 * k4 + 0] = prelu(fmaf(v[4 * k4 + 0], sc_.x, sh.x), al.x);
            v[4 * k4 + 1] = prelu(fmaf(v[4 * k4 + 1], sc_.y, sh.y), al.y);
            v[4 * k4 + 2] = prelu(fmaf(v[4 * k4 + 2], sc_.z, sh.z), al.z);
            v[4 * k4 + 3] = prelu(fmaf(v[4 * k4 + 3], sc_.w, sh.w), al.w);
          }
        }

        int r_out = q + DIL * (n0 + m);
        if (POOL == 1) {
          if (real) {
            float* xw = s_xch + (((t & 1) * 4 + grp) * 4 + q4) * 32;
            if (lane < DIL) {
#pragma unroll
              for (int k4 = 0; k4 < CW / 4; ++k4)
                *reinterpret_cast<float4*>(xw + lane * 16 + 4 * k4) = make_float4(v[4 * k4], v[4 * k4 + 1], v[4 * k4 + 2], v[4 * k4 + 3]);
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
            const bool edge = lane >= 32 - DIL;
            const float* xr = s_xch + (((t & 1) * 4 + grp) * 4 + ((q4 + 1) & 3)) * 32 + (edge ? (lane - (32 - DIL)) * 16 : 0);
#pragma unroll
            for (int k4 = 0; k4 < CW / 4; ++k4) {
              const float4 x4 = *reinterpret_cast<const float4*>(xr + 4 * k4);
              const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float nb = __shfl_down_sync(0xffffffffu, v[4 * k4 + k], DIL);
                if (edge) nb = xs[k];
                const float h = fmaxf(v[4 * k4 + k], nb);
                v[4 * k4 + k] = fmaxf(h, hprev[4 * k4 + k]);
                hprev[4 * k4 + k] = h;
              }
            }
          }
          if (m == 0) continue;
          r_out -= DIL;
        }
        if (POOL == 2) {
          // 2x2 stride-2 max-pool: pixel pairs (2j, 2j+1) never straddle a lane quarter, row pairs (2k, 2k+1) lie inside
          // an item (segments start on even rows); even lanes hold the pooled pixel j = px / 2 after an odd row
          if (real) {
#pragma unroll
            for (int k = 0; k < CW; ++k) {
              const float h = fmaxf(v[k], __shfl_down_sync(0xffffffffu, v[k], 1));
              v[k] = fmaxf(h, hprev[k]);
              hprev[k] = (m & 1) ? 0.f : h;
            }
          }
          if (!(m & 1)) continue;                  // block-uniform
          r_out >>= 1;
        }
        if constexpr (STATS) {
          if (a.stats && real) {
            const int wpx = w0 + px;
            if (wpx < a.Pw && (wpx & (a.st_pitch - 1)) < a.st_H && r_out < a.st_H) {
#pragma unroll
              for (int k = 0; k < CW; ++k) { st_s[k] += v[k]; st_q[k] = fmaf(v[k], v[k], st_q[k]); }
            }
          }
        }
        uint8_t* ob = sOut + (e % (uint32_t)a.out_bufs) * OB_BYTES;
        if (a.out_bufs == 1) {
          if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync 5, 512;" ::: "memory");
        }
        if (real) {
          uint32_t hi[CW / 2], lo[CW / 2];
#pragma unroll
          for (int k = 0; k < CW / 2; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
#pragma unroll
          for (int c = 0; c < CW / 8; ++c) {
            if (!writer) break;
            *reinterpret_cast<uint4*>(ob + row_off + (((hi_chunk + c) ^ sw) << 4)) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
            *reinterpret_cast<uint4*>(ob + 16384 + row_off + (((hi_chunk + c) ^ sw) << 4)) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        if (a.out_bufs == 2 && issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        asm volatile("bar.sync 6, 512;" ::: "memory");
        if (issuer) {
          tma_store_3d(&mapO, ob, 0, POOL == 2 ? w0 >> 1 : w0, r_out);
          tma_store_3d(&mapO, ob + 16384, 64, POOL == 2 ? w0 >> 1 : w0, r_out);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        ++e;
      }
    }
    if (t > 0)
      for (int h = 0; h < 2; ++h) sweep_drain<CW, true>(afull, aempty, dj, dph, a.S, a.bn, tcol, real, false, lane, v, timed, w_tfull);
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if constexpr (STATS) {
      if (a.stats) sweep_stats_flush<CW>(st_s, st_q, s_xch, ew, c0, real, lane, a.stats);
    }
    if (a.dbg && threadIdx.x == 64) {
      a.dbg[blockIdx.x * 8 + 5] = (unsigned long long)w_tfull; a.dbg[blockIdx.x * 8 + 6] = (unsigned long long)(clock64() - tstart);
      a.dbg[blockIdx.x * 8 + 7] = t;
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

// ---------------------------------------------------------------------------------------------------
// conv1 (1 -> 20 channels, cnn_cort/nets.py:171) straight from the volume (zero padding implicit) or from a stack of
// patches into a wide-row F32CH map.  HBM-write bound (128 B per pixel): one thread computes one pixel's 20 channels and
// writes them as three hi and three lo 16 B chunks into a SWIZZLE_128B shared tile of 256 pixels = a box of 32 x 8
// (cols x slices, or slices x cols when the SLICE axis is the contiguous one of the volume, so that the nine input loads
// of a warp stay coalesced); one TMA tensor store per tile, two tiles in flight.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

__global__ void __launch_bounds__(256) conv1_wide_kernel(const __grid_constant__ CUtensorMap mapO, const __grid_constant__ Conv1Consts cw,
                                                         const float* __restrict__ vol, ViewGeo g, int ns, int outR, int outC, int slice_fast) {
  // the 180 taps and 60 epilogue constants are kernel parameters: constant-bank operands of the FFMAs, no loads at all
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tiles = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 2 x 32 KB
  const int bc = slice_fast ? 8 : 32, bs = slice_fast ? 32 : 8;
  const int nct = (outC + bc - 1) / bc, nst = (ns + bs - 1) / bs;
  const long long n_tiles = (long long)outR * nst * nct;
  const int f = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int cl = slice_fast ? sl : f, sloc = slice_fast ? f : sl;
  const int trow = sloc * bc + cl;                                   // tile row of this thread's pixel (box order: col fastest)
  const uint32_t row_off = (uint32_t)trow * 128u, swz = (uint32_t)(trow & 7);
  uint32_t it = 0;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
    const int ct = (int)(t % nct);
    const int stl = (int)((t / nct) % nst);
    const int i = (int)(t / ((long long)nct * nst));
    const int j = ct * bc + cl, s = stl * bs + sloc;
    uint8_t* ob = tiles + (it & 1) * 32768;
    if (it >= 2) {                                                   // the store issued two tiles ago has read this buffer
      if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      __syncthreads();
    }
    float v[20];
    if (j < outC && s < ns) {
      const float* vb = vol + (int64_t)(g.s0 + s) * g.ss;
      float x[9];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int rr = g.r0 + i + ky - 16;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int cc = g.c0 + j + kx - 16;
          x[ky * 3 + kx] = (rr >= 0 && rr < g.R && cc >= 0 && cc < g.C) ? __ldg(vb + (int64_t)rr * g.rs + (int64_t)cc * g.cs) : 0.f;
        }
      }
#pragma unroll
      for (int co = 0; co < 20; ++co) {
        float acc = 0.f;
#pragma unroll
        for (int tp = 0; tp < 9; ++tp) acc = fmaf(x[tp], cw.w[tp * 20 + co], acc);
        v[co] = prelu(fmaf(acc, cw.scale[co], cw.shift[co]), cw.alpha[co]);
      }
    } else {
#pragma unroll
      for (int co = 0; co < 20; ++co) v[co] = 0.f;
    }
    uint32_t hi[12], lo[12];
#pragma unroll
    for (int k = 0; k < 10; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
    hi[10] = hi[11] = lo[10] = lo[11] = 0u;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      *reinterpret_cast<uint4*>(ob + row_off + (((uint32_t)c ^ swz) << 4)) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
      *reinterpret_cast<uint4*>(ob + row_off + (((uint32_t)(4 + c) ^ swz) << 4)) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
    }
    *reinterpret_cast<uint4*>(ob + row_off + ((3u ^ swz) << 4)) = make_uint4(0u, 0u, 0u, 0u);   // channels 24..31 stay zero
    *reinterpret_cast<uint4*>(ob + row_off + ((7u ^ swz) << 4)) = make_uint4(0u, 0u, 0u, 0u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
      tma_store_4d(&mapO, ob, 0, ct * bc, stl * bs, i);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
  if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

int launch_conv1_wide(sc_ctx* ctx, const float* vol, const ViewGeo& g, int ns, const Conv1Consts& cw, float* out, int outR, int outC,
                      cudaStream_t st) {
  TcState* s = reinterpret_cast<TcState*>(ctx->tc_state);
  SC_CHECK(s != nullptr, SC_ERR_UNSUPPORTED, "tcgen05 back-end not initialised");
  if (ns <= 0 || outR <= 0 || outC <= 0) return SC_OK;
  const int slice_fast = (g.ss == 1 && g.cs != 1) ? 1 : 0;          // axial view of a volume: z (the slice axis) is contiguous
  const int bc = slice_fast ? 8 : 32, bs = slice_fast ? 32 : 8;
  CUtensorMap mapO;
  cuuint64_t dims[4] = {64, (cuuint64_t)outC, (cuuint64_t)ns, (cuuint64_t)outR};
  cuuint64_t strides[3] = {128, (cuuint64_t)outC * 128, (cuuint64_t)ns * outC * 128};
  cuuint32_t box[4] = {64, (cuuint32_t)bc, (cuuint32_t)bs, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = s->encode(&mapO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, out, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "conv1_wide: cuTensorMapEncodeTiled failed with %d", (int)r);
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(conv1_wide_kernel), 2 * 32768 + 1024));
  const long long n_tiles = (long long)outR * ((ns + bs - 1) / bs) * ((outC + bc - 1) / bc);
  const long long cap = (long long)ctx->sm_count * 3;               // 3 CTAs per SM (66 KB of shared memory each)
  const unsigned grid = (unsigned)(n_tiles < cap ? n_tiles : cap);
  ProfScope prof(ctx, PC_CONV1, st);
  conv1_wide_kernel<<<grid, 256, 2 * 32768 + 1024, st>>>(mapO, cw, vol, g, ns, outR, outC, slice_fast);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
template <int KSTEPS, int DIL, int POOL, int CW, bool LO64, bool OUT32>
static int launch_sweep_t(sc_ctx* ctx, const CUtensorMap& mapA, const CUtensorMap& mapW, const CUtensorMap& mapO, const SweepArgs& a,
                          size_t smem, cudaStream_t st) {
  auto kern = conv_sweep_kernel<KSTEPS, DIL, POOL, CW, LO64, OUT32>;
  SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), 227 * 1024));
  const int grid = a.n_items < ctx->sm_count ? a.n_items : ctx->sm_count;
  kern<<<grid, 576, smem, st>>>(mapA, mapW, mapO, a);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// ---------------------------------------------------------------------------------------------------
// Sparse candidate masks (crop mode, brain masks): which items of a sweep does any candidate need?
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) view_occupancy_kernel(const uint8_t* __restrict__ cand, ViewGeo g, uint32_t* __restrict__ occ) {
  const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);       // one warp per (row, slice)
  if (w >= (int64_t)g.br * g.ns) return;
  const int lane = threadIdx.x & 31;
  const int i = (int)(w / g.ns), sl = (int)(w - (int64_t)i * g.ns);
  const uint8_t* base = cand + (int64_t)(g.s0 + sl) * g.ss + (int64_t)(g.r0 + i) * g.rs + (int64_t)g.c0 * g.cs;
  uint32_t bits = 0;
  for (int jb = 0; jb * 32 < g.bc; ++jb) {
    const int j = jb * 32 + lane;
    const bool on = j < g.bc && base[(int64_t)j * g.cs] != 0;
    if (__any_sync(0xffffffffu, on)) bits |= 1u << jb;
  }
  if (lane == 0) occ[w] = bits;
}

int launch_view_occupancy(sc_ctx* ctx, const uint8_t* cand, const ViewGeo& g, uint32_t* occ, cudaStream_t st) {
  SC_CHECK(g.bc <= 1024, SC_ERR_ARG, "sweep skip: more than 1024 columns per slice");
  const int64_t warps = (int64_t)g.br * g.ns;
  view_occupancy_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(cand, g, occ);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

// one warp per item (strip or strip pair x dilation class x row segment): same decoding as the sweep kernels
__global__ void __launch_bounds__(256) sweep_item_flags_kernel(const uint32_t* __restrict__ occ, int br, int bc, int ns, int C1, int reach, int n_items,
                                                               int nstr, int dil, int L, int R, int item_w, int Pw, uint8_t* __restrict__ flags) {
  const int item = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (item >= n_items) return;
  const int lane = threadIdx.x & 31;
  const int strip = item % nstr, rest = item / nstr;
  const int q = rest % dil, seg = rest / dil;
  const int Nq = (R - q + dil - 1) / dil;
  const int n0 = seg * L;
  const int Lc = Nq - n0 < L ? Nq - n0 : L;
  bool any = false;
  if (Lc > 0) {
    const int rlo = q + dil * n0, rhi = q + dil * (n0 + Lc - 1);
    const int ilo = rlo - reach > 0 ? rlo - reach : 0, ihi = rhi < br - 1 ? rhi : br - 1;
    const int w0 = strip * item_w;
    int w1 = w0 + item_w - 1;
    if (w1 > Pw - 1) w1 = Pw - 1;
    if (w0 <= w1 && ilo <= ihi) {
      const int sa = w0 / C1, sb = w1 / C1;
      const int nrow = ihi - ilo + 1;
      for (int e = lane; e < nrow * (sb - sa + 1); e += 32) {
        const int sl = sa + e / nrow, i = ilo + e % nrow;
        if (sl >= ns) continue;
        const int clo = w0 - sl * C1 > 0 ? w0 - sl * C1 : 0;
        const int chi = w1 - sl * C1 < C1 - 1 ? w1 - sl * C1 : C1 - 1;
        const int jlo = clo - reach > 0 ? clo - reach : 0, jhi = chi < bc - 1 ? chi : bc - 1;
        if (jlo > jhi) continue;
        const int b0 = jlo >> 5, b1 = jhi >> 5;
        const uint32_t colmask = (b1 - b0 == 31 ? 0xffffffffu : ((1u << (b1 - b0 + 1)) - 1u)) << b0;
        if (occ[(int64_t)i * ns + sl] & colmask) any = true;
      }
    }
  }
  any = __any_sync(0xffffffffu, any);
  if (lane == 0) flags[item] = any ? 1 : 0;
}

// fills skip->flags for the item decomposition in `a` (nstr strips or strip pairs of item_w wide columns each)
static int launch_item_flags(sc_ctx* ctx, const SweepSkip* skip, SweepArgs& a, int nstr, int item_w, int dil, int rows_out, cudaStream_t st) {
  if (!skip) return SC_OK;
  sweep_item_flags_kernel<<<(unsigned)((a.n_items + 7) / 8), 256, 0, st>>>(skip->occ, skip->br, skip->bc, skip->ns, skip->C1, rows_out - skip->br,
                                                                         a.n_items, nstr, dil, a.L, a.R, item_w, a.Pw, skip->flags);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  a.item_on = skip->flags;
  return SC_OK;
}

int launch_conv_sweep(sc_ctx* ctx, const SweepW& w, int layer, const float* in, int in_fmt, float* out, int out_fmt,
                      int Pw, int R, int rows_out, int dil, int pool, int prof_cls, cudaStream_t st, int in_dx, int in_dy, const SweepSkip* skip,
                      const SweepStats* stats) {
  TcState* s = reinterpret_cast<TcState*>(ctx->tc_state);
  SC_CHECK(s != nullptr, SC_ERR_UNSUPPORTED, "tcgen05 back-end not initialised");
  if (Pw <= 0 || R <= 0) return SC_OK;
  SweepArgs a;
  if (rows_out <= 0 || rows_out > R) rows_out = R;                      // rows of the map the next layer actually reads
  a.Pw = Pw; a.R = rows_out; a.bn = w.bn;
  a.strip_w = 128 - (pool == 1 ? dil : 0);                            // pool: 0 none, 1 stride-1 window {0,d}^2, 2 = 2x2 stride 2
  a.nstrips = (Pw + a.strip_w - 1) / a.strip_w;
  const int nq = (rows_out + dil - 1) / dil;                            // class rows of the largest class
  // segments: enough items to balance the SMs, rows per item long enough to amortise the 2 (+1) halo rows
  int nseg = (4 * ctx->sm_count + a.nstrips * dil - 1) / (a.nstrips * dil);
  int L = (nq + nseg - 1) / nseg;
  if (L < 12) L = 12;
  if (a.nstrips * dil * ((nq + 11) / 12) < ctx->sm_count) {            // small maps (training batches): 12-row items would leave SMs idle,
    nseg = (ctx->sm_count + a.nstrips * dil - 1) / (a.nstrips * dil);  // so the rows are cut finer (down to 2 per item) to fill the machine once
    L = (nq + nseg - 1) / nseg;
    if (L < 2) L = 2;
  }
  if (L > 96) L = 96;
  if (skip && L > 32) L = 32;                                           // sparse candidate mask: finer items skip more
  if (pool == 2) L = (L + 1) & ~1;                                      // row pairs of the stride-2 pool stay inside an item
  nseg = (nq + L - 1) / L;
  a.L = L; a.nseg = nseg;
  a.n_items = a.nstrips * dil * nseg;
  a.item_on = nullptr;
  a.stats = nullptr; a.st_H = 0; a.st_pitch = 1;
  if (stats) {
    SC_CHECK(dil == 1 && !pool && (stats->pitch & (stats->pitch - 1)) == 0, SC_ERR_ARG, "conv_sweep: fused statistics need dil 1, no pool, a power-of-two pitch");
    a.stats = stats->sums; a.st_H = stats->H; a.st_pitch = stats->pitch;
  }
  SC_CHECK(pool != 2 || dil == 1, SC_ERR_ARG, "conv_sweep: the stride-2 pool needs dilation 1");
  a.npanels = w.npanels;
  a.in_dx = in_dx; a.in_dy = in_dy;
  a.scale = w.scale; a.shift = w.shift; a.alpha = w.alpha;
  a.dbg = (ctx->tc_timing_cls == prof_cls) ? ctx->tc_timing_buf : nullptr;
  SC_CHECK(w.bn <= (out_fmt ? 32 : 64) && w.bn % 16 == 0, SC_ERR_ARG, "conv_sweep: bad channel geometry");
  a.S = 512 / w.bn - 2;                                                 // accumulator slots + 2 spill slots fill the 512 TMEM columns
  if (a.S > SW_MAX_SLOTS) a.S = SW_MAX_SLOTS;
  const int slot = (in_fmt ? 1 : 2) * SW_SLOT_HALF;                      // F32CH: one box per row (hi|lo in one 128 B pixel), F64CH: hi box + lo box
  const int w_bytes = w.npanels * 6 * w.bn * 128;
  const int ob_bytes = out_fmt ? 16384 : 32768;
  const int fixed = 1024 + w_bytes + SW_BAR_BYTES + 192 * 4 + 2 * 4 * 4 * 2 * 16 * 4;
  // ring: one stage per input row in the MMAs, the others prefetch; two output tiles if that leaves >= 3 stages
  a.out_bufs = 2;
  a.stages = (227 * 1024 - fixed - 2 * ob_bytes) / slot;
  if (a.stages < 3) {                                                   // short of shared memory: single output tile
    a.out_bufs = 1;
    a.stages = (227 * 1024 - fixed - ob_bytes) / slot;
  }
  if (a.stages > 8) a.stages = 8;
  const bool use_pair = w.ksteps >= 3 && !in_fmt && !out_fmt;          // >= 40 input channels: the resident weights need the CTA pair
  SC_CHECK(use_pair || a.stages >= 2, SC_ERR_ARG, "conv_sweep: ring does not fit (layer %d)", layer);
  const size_t smem = (size_t)fixed + (size_t)a.stages * slot + (size_t)a.out_bufs * ob_bytes;

  CUtensorMap mapA, mapW, mapO;
  {
    const int pxe = in_fmt ? 64 : 128;                                    // bf16 elements per pixel
    cuuint64_t dims[3] = {(cuuint64_t)pxe, (cuuint64_t)Pw, (cuuint64_t)R};
    cuuint64_t strides[2] = {(cuuint64_t)pxe * 2, (cuuint64_t)Pw * pxe * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)(128 + 2 * dil), 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = s->encode(&mapA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<float*>(in), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "conv_sweep: cuTensorMapEncodeTiled(A) failed with %d (Pw %d R %d)", (int)r, Pw, R);
  }
  {
    cuuint64_t dims[2] = {64, (cuuint64_t)w.npanels * 6 * w.bn};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {64, (cuuint32_t)(3 * w.bn)};                    // W hi or W lo rows of one panel (<= 192 rows)
    cuuint32_t es[2] = {1, 1};
    CUresult r = s->encode(&mapW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.panels, dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "conv_sweep: cuTensorMapEncodeTiled(W) failed with %d", (int)r);
  }
  {
    // output: one box of strip_w pixels x 128 B per store (hi and lo boxes for the 256 B pixels); the columns a strip
    // does not own (pool reach) are simply not part of the box
    const int pxe = out_fmt ? 64 : 128;
    const int oPw = pool == 2 ? Pw / 2 : Pw, oR = pool == 2 ? R / 2 : R;   // stride-2 pool: pitch and rows halve
    cuuint64_t dims[3] = {(cuuint64_t)pxe, (cuuint64_t)oPw, (cuuint64_t)oR};
    cuuint64_t strides[2] = {(cuuint64_t)pxe * 2, (cuuint64_t)oPw * pxe * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)(pool == 2 ? 64 : a.strip_w), 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = s->encode(&mapO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, out, dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "conv_sweep: cuTensorMapEncodeTiled(O) failed with %d", (int)r);
  }
  const bool i32 = in_fmt != 0, o32 = out_fmt != 0;
  if (use_pair) {
    // ---- CTA pairs: half of the weights per CTA ----
    const int nsp = (a.nstrips + 1) / 2;
    const int pairs_max = ctx->sm_count / 2;
    nseg = (4 * pairs_max + nsp * dil - 1) / (nsp * dil);
    L = (nq + nseg - 1) / nseg;
    if (L < 12) L = 12;
    if (nsp * dil * ((nq + 11) / 12) < pairs_max) {
      nseg = (pairs_max + nsp * dil - 1) / (nsp * dil);
      L = (nq + nseg - 1) / nseg;
      if (L < 2) L = 2;
    }
    if (L > 96) L = 96;
    if (skip && L > 32) L = 32;
    if (pool == 2) L = (L + 1) & ~1;
    nseg = (nq + L - 1) / L;
    a.L = L; a.nseg = nseg;
    a.n_items = nsp * dil * nseg;
    const int wp_bytes = w.npanels * 3 * w.bn * 128;
    const int fixed_p = 1024 + ((wp_bytes + 1023) & ~1023) + SW_BAR_BYTES + 192 * 4 + ((pool || stats) ? 2 * 4 * 4 * 2 * 16 * 4 : 0);
    a.out_bufs = 2;
    a.stages = (227 * 1024 - fixed_p - 2 * ob_bytes) / slot;
    if (a.stages < 3) { a.out_bufs = 1; a.stages = (227 * 1024 - fixed_p - ob_bytes) / slot; }
    if (a.stages > 8) a.stages = 8;
    SC_CHECK(a.stages >= 2, SC_ERR_ARG, "conv_sweep: pair ring does not fit (layer %d)", layer);
    SC_CHECK(pool != 2 || (Pw % 2 == 0), SC_ERR_ARG, "conv_sweep: odd pitch with the stride-2 pool");
    const size_t smem_p = (size_t)fixed_p + (size_t)a.stages * slot + (size_t)a.out_bufs * ob_bytes;
    CUtensorMap mapWp;
    cuuint64_t dims[2] = {64, (cuuint64_t)w.npanels * 6 * w.bn};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {64, (cuuint32_t)(3 * w.bn)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = s->encode(&mapWp, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.panels_pair, dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SC_CHECK(r == CUDA_SUCCESS, SC_ERR_CUDA, "conv_sweep: cuTensorMapEncodeTiled(W pair) failed with %d", (int)r);
    const int npairs = a.n_items < pairs_max ? a.n_items : pairs_max;
    SC_TRY(launch_item_flags(ctx, skip, a, nsp, 2 * a.strip_w, dil, rows_out, st));
    ProfScope prof(ctx, prof_cls, st);
    if (dil == 1 && pool == 2) {
      auto kern = conv_sweep_pair_kernel<3, 1, 2>;
      SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), 227 * 1024));
      kern<<<2 * npairs, 576, smem_p, st>>>(mapA, mapWp, mapO, a);
    } else if (dil == 1 && !pool && w.ksteps == 4) {   // training: dgrad of conv5 (60 input channels)
      auto kern = conv_sweep_pair_kernel<4, 1, 0>;
      SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), 227 * 1024));
      kern<<<2 * npairs, 576, smem_p, st>>>(mapA, mapWp, mapO, a);
    } else if (dil == 1 && !pool) {
      auto kern = conv_sweep_pair_kernel<3, 1, 0>;
      SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), 227 * 1024));
      kern<<<2 * npairs, 576, smem_p, st>>>(mapA, mapWp, mapO, a);
    } else if (dil == 2 && pool == 1) {
      auto kern = conv_sweep_pair_kernel<3, 2, 1>;
      SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), 227 * 1024));
      kern<<<2 * npairs, 576, smem_p, st>>>(mapA, mapWp, mapO, a);
    } else if (dil == 4 && !pool) {
      auto kern = conv_sweep_pair_kernel<3, 4, 0>;
      SC_TRY(ensure_smem_attr(ctx, reinterpret_cast<const void*>(kern), 227 * 1024));
      kern<<<2 * npairs, 576, smem_p, st>>>(mapA, mapWp, mapO, a);
    } else {
      set_error("conv_sweep: no pair kernel instance for dil=%d pool=%d", dil, pool);
      return SC_ERR_ARG;
    }
    ctx->launches++;
    SC_CUDA(cudaGetLastError());
    return SC_OK;
  }
  SC_TRY(launch_item_flags(ctx, skip, a, a.nstrips, a.strip_w, dil, rows_out, st));
  ProfScope prof(ctx, prof_cls, st);
  if (w.ksteps == 2 && dil == 1 && pool == 2 && i32 && o32 && w.bn == 32) return launch_sweep_t<2, 1, 2, 8, true, true>(ctx, mapA, mapW, mapO, a, smem, st);     // patch maps: conv2 + 2x2/2 pool
  if (w.ksteps == 2 && dil == 1 && pool == 1 && i32 && o32 && w.bn == 32) return launch_sweep_t<2, 1, 1, 8, true, true>(ctx, mapA, mapW, mapO, a, smem, st);     // conv2 + pool1
  if (w.ksteps == 2 && dil == 2 && !pool && i32 && !o32) return launch_sweep_t<2, 2, 0, 16, true, false>(ctx, mapA, mapW, mapO, a, smem, st);              // conv3
  // patchwise maps (dilation 1 everywhere, stride-2 pools stay separate passes)
  if (w.ksteps == 2 && dil == 1 && !pool && i32 && !o32) return launch_sweep_t<2, 1, 0, 16, true, false>(ctx, mapA, mapW, mapO, a, smem, st);
  // training: raw conv2 forward and its dgrad (20 -> 20 channels, 128 B pixels in and out)
  if (w.ksteps == 2 && dil == 1 && !pool && i32 && o32 && w.bn == 32) return launch_sweep_t<2, 1, 0, 8, true, true>(ctx, mapA, mapW, mapO, a, smem, st);
  set_error("conv_sweep: no kernel instance for ksteps=%d dil=%d pool=%d in_fmt=%d out_fmt=%d", w.ksteps, dil, pool, in_fmt, out_fmt);
  return SC_ERR_ARG;
}

}  // namespace sc
