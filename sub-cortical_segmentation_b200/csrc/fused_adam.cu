// Gradient all-reduce fused with the Adam update in ONE kernel over NVLink peer memory (SURVEY.md 5.8, K5).
//
// Data-parallel training exchanges one flat 883 455-float gradient buffer per step (cnn_cort/nets.py:236-237 is a single
// device; the exchange is new).  Instead of ncclAllReduce followed by an update kernel on every rank, every rank
//   1. announces "my gradients are complete" to all peers (flag store into each peer's flag page, system scope) and waits for
//      theirs,
//   2. sums ITS 1/world slice of the gradients straight out of the peers' buffers (peer loads over NVLink / NVSwitch, fixed
//      rank order, so every element is reduced exactly once, by one rank) and applies Lasagne's Adam to that slice (the
//      moment buffers are only ever touched inside the owner's slice: ZeRO-1 style sharding of the optimiser state),
//   3. broadcasts the updated parameters of the slice into every peer's parameter buffer (peer stores),
//   4. announces "my slice is written everywhere" and waits for the peers, so that when the kernel retires every rank's
//      parameter buffer is complete and nobody reads this rank's gradients any more.
// All ranks end with bit-identical parameters by construction.  The buffers are exchanged once as CUDA IPC handles
// (one process per GPU).  3.5 MB per step: the cost is the two flag round trips, not bandwidth.
#include "common.cuh"

namespace sc {

struct PeerTable { float* grads[8]; float* params[8]; unsigned* flags[8]; };

__device__ __forceinline__ void st_flag(unsigned* p, unsigned v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_flag(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_peer(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

// flags page of a rank: [0 .. 8) "gradients ready" per peer, [8 .. 16) "slice written" per peer, [16] local go, [17] local arrivals
__global__ void __launch_bounds__(512) allreduce_adam_kernel(PeerTable T, int rank, int world, float* __restrict__ m, float* __restrict__ v,
                                                             const uint8_t* __restrict__ trainable, int n, float a_t, float b1, float b2,
                                                             float eps, float sscale, unsigned step) {
  unsigned* mine = T.flags[rank];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    __threadfence_system();                                  // this rank's backward pass wrote the gradients on this stream
    for (int p = 0; p < world; ++p) st_flag(T.flags[p] + rank, step);
    for (int p = 0; p < world; ++p) while (ld_flag(mine + p) < step) { }
    st_flag(mine + 16, step);                                // release the other CTAs of this grid
  }
  if (threadIdx.x == 0) while (ld_flag(mine + 16) < step) { }
  __syncthreads();

  const int chunk = (((n + world - 1) / world) + 3) & ~3;
  const int lo = rank * chunk, hi = min(n, lo + chunk);
  for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
    float g = 0.f;
    for (int p = 0; p < world; ++p) g += ld_peer(T.grads[p] + i);
    float np_;
    const float pi = T.params[rank][i];
    const uint8_t t = trainable[i];
    if (t == 1) {
      const float mi = b1 * m[i] + (1.f - b1) * g;
      const float vi = b2 * v[i] + (1.f - b2) * g * g;
      m[i] = mi; v[i] = vi;
      np_ = pi - a_t * mi / (sqrtf(vi) + eps);
    } else if (t == 0) {
      np_ = 0.9f * pi + 0.1f * (g * sscale);                 // BN running mean / inv_std: average of the ranks' batch statistics
    } else {
      np_ = pi;                                              // 2: frozen (sc_freeze_trunk)
    }
    for (int p = 0; p < world; ++p) T.params[p][i] = np_;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned arrived = atomicAdd(mine + 17, 1u) + 1u;
    if (arrived == gridDim.x * step) {                       // last CTA of this launch (the counter is never reset)
      __threadfence_system();
      for (int p = 0; p < world; ++p) st_flag(T.flags[p] + 8 + rank, step);
      for (int p = 0; p < world; ++p) while (ld_flag(mine + 8 + p) < step) { }
    }
  }
}

int fused_export(sc_ctx* ctx, unsigned char* handles /* 3 x 64 bytes */) {
  SC_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->peer_flags) {
    SC_CUDA(cudaMalloc(&ctx->peer_flags, 256));
    SC_CUDA(cudaMemset(ctx->peer_flags, 0, 256));
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  SC_CUDA(cudaIpcGetMemHandle(&h, ctx->grads)); memcpy(handles, &h, 64);
  SC_CUDA(cudaIpcGetMemHandle(&h, ctx->params)); memcpy(handles + 64, &h, 64);
  SC_CUDA(cudaIpcGetMemHandle(&h, ctx->peer_flags)); memcpy(handles + 128, &h, 64);
  return SC_OK;
}

int fused_attach(sc_ctx* ctx, int rank, int world, const unsigned char* all /* world x 3 x 64 bytes */) {
  SC_CHECK(world >= 1 && world <= 8 && rank >= 0 && rank < world, SC_ERR_ARG, "sc_fused_attach: world must be 1..8");
  SC_CHECK(ctx->peer_flags != nullptr, SC_ERR_STATE, "sc_fused_attach: call sc_fused_export first");
  SC_CUDA(cudaSetDevice(ctx->device));
  for (int p = 0; p < world; ++p) {
    if (p == rank) {
      ctx->peer_grads[p] = ctx->grads; ctx->peer_params[p] = ctx->params; ctx->peer_flagp[p] = ctx->peer_flags;
      continue;
    }
    cudaIpcMemHandle_t h;
    void* ptr = nullptr;
    memcpy(&h, all + (size_t)p * 192, 64);
    SC_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess)); ctx->peer_grads[p] = reinterpret_cast<float*>(ptr);
    memcpy(&h, all + (size_t)p * 192 + 64, 64);
    SC_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess)); ctx->peer_params[p] = reinterpret_cast<float*>(ptr);
    memcpy(&h, all + (size_t)p * 192 + 128, 64);
    SC_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess)); ctx->peer_flagp[p] = reinterpret_cast<unsigned*>(ptr);
  }
  ctx->peer_rank = rank; ctx->peer_world = world;       // (peer_step keeps counting: the flag pages are never reset)
  return SC_OK;
}

void fused_detach(sc_ctx* ctx) {
  for (int p = 0; p < ctx->peer_world; ++p) {
    if (p == ctx->peer_rank) continue;
    if (ctx->peer_grads[p]) cudaIpcCloseMemHandle(ctx->peer_grads[p]);
    if (ctx->peer_params[p]) cudaIpcCloseMemHandle(ctx->peer_params[p]);
    if (ctx->peer_flagp[p]) cudaIpcCloseMemHandle(ctx->peer_flagp[p]);
  }
  ctx->peer_world = 0;
  if (ctx->peer_flags) { cudaFree(ctx->peer_flags); ctx->peer_flags = nullptr; }
}

int fused_allreduce_adam(sc_ctx* ctx, float lr, float b1, float b2, float eps, cudaStream_t st) {
  SC_CHECK(ctx->peer_world >= 1, SC_ERR_STATE, "sc_allreduce_adam_step: call sc_fused_attach first");
  ctx->adam_t += 1;
  ctx->peer_step += 1;
  const double t = (double)ctx->adam_t;
  const float a_t = (float)(lr * sqrt(1.0 - pow((double)b2, t)) / (1.0 - pow((double)b1, t)));
  PeerTable T;
  for (int p = 0; p < 8; ++p) { T.grads[p] = ctx->peer_grads[p]; T.params[p] = ctx->peer_params[p]; T.flags[p] = ctx->peer_flagp[p]; }
  ProfScope prof(ctx, PC_ADAM, st);
  // few enough CTAs to be co-resident (the grid spins on flags): the slice is at most 883 455 floats
  allreduce_adam_kernel<<<32, 512, 0, st>>>(T, ctx->peer_rank, ctx->peer_world, ctx->adam_m, ctx->adam_v, ctx->trainable, SC_PARAM_FLOATS, a_t, b1,
                                            b2, eps, 1.f / (float)ctx->peer_world, ctx->peer_step);
  ctx->launches++;
  ctx->derived_dirty = true;
  SC_CUDA(cudaGetLastError());
  return SC_OK;
}

}  // namespace sc
