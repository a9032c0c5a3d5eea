// Training-time augmentation inside the minibatch gather (sc_gather_samples_augmented, contract in the header): per sample one
// random similarity M = s R about the centre voxel, trilinear sampling of the zero-extended scan, then contrast, brightness and
// Gaussian noise.  Random numbers come from hash3 keyed by (seed, epoch, table row), so the kernel needs no state.
#include <math.h>

#include "common.cuh"

namespace sc {

constexpr uint64_t kEpochMix = 0xD1B54A32D192ED03ull;
constexpr int kAugSlots = 8192;     // hash slots per row: 0..5 the sample's parameters, 1024.. the per-pixel noise pairs
constexpr int kNoiseSlot = 1024;

__device__ __forceinline__ double aug_u(uint64_t se, uint64_t key) { return ((double)hash3(se, key) + 0.5) * 0x1p-32; }

// ln u of u = (h + 0.5) 2^-32 to float precision over the whole of (0, 1): log of u below 1/2, log1p of -(1 - u) above
__device__ __forceinline__ float aug_log_u(uint32_t h) {
  if (h < 0x80000000u) return logf(((float)h + 0.5f) * 0x1p-32f);
  return log1pf(-(((float)(0xFFFFFFFFu - h) + 0.5f) * 0x1p-32f));
}

// Same work decomposition as gather_samples_kernel: one warp per (sample, view), lane = patch column j, a loop over the 32
// patch rows, every store one full 128 B patch row.  A rotated patch has no contiguous axis, so each pixel's 8 corner loads are
// scattered sectors; neighbouring pixels share most of them through L1 / L2.  The three warps of a sample derive M, a and b
// from the same hashes.
__global__ void __launch_bounds__(256) gather_samples_augmented_kernel(
    const sc_scan* __restrict__ scans, int n_scans, const int32_t* __restrict__ samples, const float* __restrict__ atlas_rows,
    const uint8_t* __restrict__ labels, const int64_t* __restrict__ idx, int64_t n, sc_augment aug, float* __restrict__ ax,
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
  // an invalid scan index reads as an empty volume (every corner outside), never an out-of-bounds access
  const float* vol = nullptr;
  int X = 0, Y = 0, Z = 0;
  if ((unsigned)row.x < (unsigned)n_scans) {
    vol = scans[row.x].vol;
    X = scans[row.x].dims[0]; Y = scans[row.x].dims[1]; Z = scans[row.x].dims[2];
  }
  const int64_t YZ = (int64_t)Y * Z;

  // ---- the sample's transform, in double, rounded to float
  const uint64_t se = aug.seed ^ ((uint64_t)aug.epoch * kEpochMix);
  const uint64_t key = (uint64_t)r * kAugSlots;
  const double kz = 2.0 * aug_u(se, key + 0) - 1.0;
  const double kr = sqrt(fmax(0.0, 1.0 - kz * kz));
  double sphi, cphi;
  sincospi(2.0 * aug_u(se, key + 1), &sphi, &cphi);
  const double k0 = kr * cphi, k1 = kr * sphi, k2 = kz;
  double st, ct;
  sincospi((double)aug.rotation_deg * (2.0 * aug_u(se, key + 2) - 1.0) / 180.0, &st, &ct);
  const double scl = pow(1.0 + (double)aug.scale, 2.0 * aug_u(se, key + 3) - 1.0);
  const float a = (float)(1.0 + (double)aug.intensity * (2.0 * aug_u(se, key + 4) - 1.0));
  const float b = (float)((double)aug.intensity * (2.0 * aug_u(se, key + 5) - 1.0));
  // Rodrigues: R = cos(t) I + sin(t) [k]x + (1 - cos(t)) k k^T; the view needs the columns of its row and column axes
  const double vc = 1.0 - ct;
  const double R[3][3] = {{ct + vc * k0 * k0, -st * k2 + vc * k0 * k1, st * k1 + vc * k0 * k2},
                          {st * k2 + vc * k1 * k0, ct + vc * k1 * k1, -st * k0 + vc * k1 * k2},
                          {-st * k1 + vc * k2 * k0, st * k0 + vc * k2 * k1, ct + vc * k2 * k2}};
  float mr[3], mc[3];   // M e_row, M e_col: axial rows x, cols y; coronal rows x, cols z; saggital rows y, cols z
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    mr[q] = (float)(scl * (view == 2 ? R[q][1] : R[q][0]));
    mc[q] = (float)(scl * (view == 0 ? R[q][1] : R[q][2]));
  }

  // ---- the patch: p = c + (i - 16) M e_row + (j - 16) M e_col
  const float jo = (float)(lane - 16);
  const float q0 = fmaf(jo, mc[0], (float)row.y), q1 = fmaf(jo, mc[1], (float)row.z), q2 = fmaf(jo, mc[2], (float)row.w);
  const bool noisy = aug.noise > 0.f;
  float* out = dst + s * 1024 + lane;
  for (int i = 0; i < 32; ++i) {
    const float io = (float)(i - 16);
    const float px = fmaf(io, mr[0], q0), py = fmaf(io, mr[1], q1), pz = fmaf(io, mr[2], q2);
    const float fx = floorf(px), fy = floorf(py), fz = floorf(pz);
    const float tx = px - fx, ty = py - fy, tz = pz - fz;
    const int ix = (int)fx, iy = (int)fy, iz = (int)fz;
    const bool vx[2] = {ix >= 0 && ix < X, ix + 1 >= 0 && ix + 1 < X};
    const bool vy[2] = {iy >= 0 && iy < Y, iy + 1 >= 0 && iy + 1 < Y};
    const bool vz[2] = {iz >= 0 && iz < Z, iz + 1 >= 0 && iz + 1 < Z};
    const float wx[2] = {1.f - tx, tx}, wy[2] = {1.f - ty, ty}, wz[2] = {1.f - tz, tz};
    const int64_t base = (int64_t)ix * YZ + (int64_t)iy * Z + iz;
    float acc = 0.f;
#pragma unroll
    for (int dx = 0; dx < 2; ++dx)
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dz = 0; dz < 2; ++dz) {
          const float v = vx[dx] && vy[dy] && vz[dz] ? __ldg(vol + base + dx * YZ + (int64_t)dy * Z + dz) : 0.f;
          acc = fmaf(wx[dx] * wy[dy] * wz[dz], v, acc);
        }
    float val = fmaf(a, acc, b);
    if (noisy) {
      const uint64_t nk = key + kNoiseSlot + 2 * (uint64_t)(view * 1024 + i * 32 + lane);
      const float g = sqrtf(-2.f * aug_log_u(hash3(se, nk))) * cospif(2.f * (((float)hash3(se, nk + 1) + 0.5f) * 0x1p-32f));
      val = fmaf(aug.noise, g, val);
    }
    __stcs(out, val);
    out += 32;
  }
}

int launch_gather_samples_augmented(sc_ctx* ctx, const sc_scan* scans, int n_scans, const int32_t* samples, const float* atlas_rows,
                                    const uint8_t* labels, const int64_t* idx, int64_t n, const sc_augment& aug, float* ax, float* co,
                                    float* sa, float* atlas_out, uint8_t* y_out, cudaStream_t st) {
  if (n == 0) return SC_OK;
  const int64_t blocks = (n * 3 + 7) / 8;
  SC_CHECK(blocks < (1ll << 31), SC_ERR_ARG, "sc_gather_samples_augmented: too many samples in one call");
  ProfScope prof(ctx, PC_AUGMENT, st);
  gather_samples_augmented_kernel<<<(unsigned)blocks, 256, 0, st>>>(scans, n_scans, samples, atlas_rows, labels, idx, n, aug, ax, co,
                                                                    sa, atlas_out, y_out);
  ctx->launches++;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
