// kernels_dp.cuh -- data-parallel gradient exchange fused with the optimizer, over NVLink peer memory.
//
// The data-parallel large-batch mode (BASELINE config 5; mr_gan.py:165-167 is the update being distributed) needs, once per
// D or G step, sum-over-ranks of the flat gradient followed by Keras Adam on every parameter.  The NCCL path (a handle
// whose IPC handles were not opened) all-reduces the whole gradient (2 (W-1)/W x 4 B per parameter over the links) and
// then every rank runs the full Adam (28 B per parameter of HBM traffic on EVERY rank).  k_dp_exchange does both in ONE
// kernel per rank:
//
//   reduce-scatter by peer LOADS : rank r owns the r-th 1/W of the flat range; it reads that shard of every rank's gradient
//                                  buffer straight out of the peers' HBM (NVLink P2P loads, summed in rank order)
//   sharded Adam                 : m, v and the fp32 master weights are read and written for the owned shard only
//                                  (28 / W B per parameter of local HBM traffic)
//   all-gather by peer STORES    : the updated weights (and, in f16 mode, their fp16 operand copies) are written into
//                                  every rank's parameter buffer
//
// so each parameter crosses the links (W-1)/W x 4 B in (gradient) and (W-1)/W x 4 B (+2) out (weights), the math rides on
// the transfers, and no rank touches optimizer state it does not own.  Cross-GPU ordering uses two flag barriers in peer
// memory ("all gradients complete" before the loads, "all weights delivered" before the kernel may finish); arrival
// flags carry a monotonically increasing sequence number kept on the device, so the kernel is CUDA-graph capturable.
// The same kernel runs the VIRTUAL-rank mode (one launch, gridDim.y = W virtual ranks over the folds of one handle,
// cooperative so that all CTAs are co-resident), which is how it is tested on one GPU.
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"

#define DP_MAX_RANKS 8
#define DP_FLAG_WORDS 32            // per rank: [0..8) arrivals A, [8..16) arrivals B, [16] sequence, [17] finished CTAs

struct DpPeers {
  float* P[DP_MAX_RANKS];           // parameter buffers (flat, identical layout on every rank)
  float* Gr[DP_MAX_RANKS];          // gradient buffers
  __half* Ph[DP_MAX_RANKS];         // fp16 operand copies of the parameters (null unless f16 mode)
  unsigned* flags[DP_MAX_RANKS];    // flag blocks (DP_FLAG_WORDS words each)
  float* Mo[DP_MAX_RANKS];          // Adam slots: only [rank] is ever touched by that rank
  float* Vo[DP_MAX_RANKS];
};

namespace dp {
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float4 ld_peer(const float4* p) {      // never served from a stale local cache line
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
// one thread: tell every rank (slot `me` of its block) that this rank reached sequence `seq`
__device__ __forceinline__ void signal_all(const DpPeers& pp, int W, int me, int base, unsigned seq) {
  __threadfence_system();
  for (int p = 0; p < W; ++p) st_release_sys(pp.flags[p] + base + me, seq);
}
// one thread: wait until every rank has signalled `seq` into MY block; a missing rank traps instead of hanging the GPU
__device__ __forceinline__ void wait_all(const unsigned* mine, int W, int base, unsigned seq) {
  for (int p = 0; p < W; ++p) {
    const long long t0 = clock64();
    while ((int)(ld_acquire_sys(mine + base + p) - seq) < 0) {
      if (clock64() - t0 > (1ll << 32)) __trap();
    }
  }
}
}  // namespace dp

// grid = (blocks per rank, virtual ranks or 1).  [off, off + len) is the flat range of the net being updated (len % 4 == 0).
// rank < 0: virtual-rank mode, the rank is blockIdx.y.  `folds` / `nfolds`: the LOCAL fold states whose counters this rank
// advances (virtual mode: fold blockIdx.y only).
__global__ void __launch_bounds__(256)
k_dp_exchange(DpPeers pp, int W, int rank, long long off, long long len, FoldState* __restrict__ folds, int nfolds, int net,
              AdamHyper hp, float ginv) {
  const bool virt = rank < 0;
  const int me = virt ? (int)blockIdx.y : rank;
  FoldState* const myfolds = virt ? folds + me : folds;
  const int nmy = virt ? 1 : nfolds;
  unsigned* const mine = pp.flags[me];
  __shared__ unsigned s_seq;
  if (threadIdx.x == 0) {
    const unsigned seq = dp::ld_acquire_sys(mine + 16) + 1u;      // every CTA is resident before the last one bumps it
    s_seq = seq;
    if (blockIdx.x == 0) dp::signal_all(pp, W, me, 0, seq);       // A: my gradient buffer is complete (kernel boundary + fence)
    dp::wait_all(mine, W, 0, seq);                                // A: everybody's is
  }
  __syncthreads();
  const unsigned seq = s_seq;

  // ---- owned shard: quads [q0, q1) of the range ----
  const long long nq = len >> 2;
  const long long q0 = nq * me / W, q1 = nq * (me + 1) / W;
  const float lr_t = myfolds[0].lr_t[net];
  const float b1 = hp.b1, b2 = hp.b2, c1 = 1.0f - hp.b1, c2 = 1.0f - hp.b2, eps = hp.eps;
  float4* const m4 = reinterpret_cast<float4*>(pp.Mo[me] + off);
  float4* const v4 = reinterpret_cast<float4*>(pp.Vo[me] + off);
  const float4* const p4 = reinterpret_cast<const float4*>(pp.P[me] + off);
  for (long long i = q0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < q1; i += (long long)gridDim.x * blockDim.x) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
    for (int p = 0; p < W; ++p) {                                 // rank order: the sum is the same whoever owns the shard
      const float4 x = dp::ld_peer(reinterpret_cast<const float4*>(pp.Gr[p] + off) + i);
      g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
    }
    g.x *= ginv; g.y *= ginv; g.z *= ginv; g.w *= ginv;
    float4 pw = p4[i], m = m4[i], v = v4[i];
#define ADAM1(c) m.c = fmaf(b1, m.c, c1 * g.c); v.c = fmaf(b2, v.c, c2 * g.c * g.c); pw.c -= lr_t * m.c / (sqrtf(v.c) + eps);
    ADAM1(x) ADAM1(y) ADAM1(z) ADAM1(w)
#undef ADAM1
    m4[i] = m; v4[i] = v;
    const __half2 h01 = __floats2half2_rn(pw.x, pw.y), h23 = __floats2half2_rn(pw.z, pw.w);
    for (int p = 0; p < W; ++p) {                                 // all-gather: the updated shard goes to every rank
      reinterpret_cast<float4*>(pp.P[p] + off)[i] = pw;
      if (pp.Ph[p]) {
        __half2* const hp2 = reinterpret_cast<__half2*>(pp.Ph[p] + off) + 2 * i;
        hp2[0] = h01; hp2[1] = h23;
      }
    }
  }
  // ---- B: my shard has been delivered everywhere; nobody's next forward may start before all shards have arrived ----
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicAdd(mine + 17, 1u) + 1u;
    if (done == gridDim.x) {                                      // the last CTA of this rank
      mine[17] = 0u;
      dp::signal_all(pp, W, me, 8, seq);
      dp::wait_all(mine, W, 8, seq);
      for (int f = 0; f < nmy; ++f) {                             // K.update_add(iterations, 1); noise step
        if (hp.shared_t) myfolds[f].iterations += 1; else myfolds[f].it_net[net] += 1;
        myfolds[f].rng_step += 1;
      }
      __threadfence_system();
      dp::st_release_sys(mine + 16, seq);
    }
  }
}
