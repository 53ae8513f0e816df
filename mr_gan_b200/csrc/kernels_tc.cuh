// kernels_tc.cuh -- tcgen05 / TMEM / TMA grouped GEMM of the training step (precision = tf32).
//
// One warp-specialised kernel serves all dense contractions of the step, grouped over folds
// (blockIdx.z) with per-(op, fold) TMA descriptors resident in HBM:
//
//   role            MMA-A (M = 128 "feature" rows)          MMA-B (N = bn columns)            accumulator
//   forward         W^T  from Waug[k, n]  (MN-major)        act  from A[r, k]   (K-major)     D[n, r]
//   backward dX     W    from Waug[k, n]  (K-major)         dZ   from dZ[r, n]  (K-major)     D[k, r]
//   backward dW     dZ^T from dZ[r, n]    (MN-major)        A^T  from A[r, k]   (MN-major)    D[n, k]
//
// i.e. the weight-side dimension always sits on the 128 TMEM lanes ("swap-AB": the batch is only
// 50..150 rows, mr_gan.py:78) and fp32 master weights feed kind::tf32 MMAs directly -- no low
// precision shadow copy, no transposed copy (both operand majors are legal for tf32 descriptors).
// The lane <-> memory-contiguous-dimension match makes every epilogue access coalesced:
// thread = one feature, registers = rows (forward / dX) or input features (dW).
//
// Pipeline: warp 0 = TMA producer (4-stage mbarrier ring, 32 contraction elements per stage),
// warp 1 = TMEM allocator + single-thread tcgen05.mma issuer, warps 2..5 = epilogue
// (tcgen05.ld 32x32b -> bias-free activation + Philox GaussianNoise | act' mask | dW store).
#pragma once
#include <cuda.h>
#include "common.cuh"

// Reductions fused into the epilogue of the GEMM that produces their input (thread = feature, the batch is in TMEM columns,
// so batch statistics are thread-local):
//   HEAD_DISC    forward of the logit layer: Salimans supervised / unsupervised losses, training error, logit gradients
//                (mr_gan.py:146-149,161), and K.update_add(iterations, 1) of the discriminator step
//   HEAD_FM      forward of D layer 5 in the generator step: feature-matching loss and its gradient (mr_gan.py:152-154)
//   HEAD_BN      forward of G layer 1: BatchNormalization with batch statistics (mr_gan.py:112)
enum { HEAD_NONE = 0, HEAD_DISC = 1, HEAD_FM = 2, HEAD_BN = 3 };

struct alignas(64) TcOp {
  CUtensorMap mapA, mapB;
  GemmDesc g;                 // epilogue description shared with the fp32 path (C, C2, aux, act, noise ...)
  int ME, NE, KE;             // extents: MMA-M (features), MMA-N, contraction
  int bn;                     // MMA-N per tile (multiple of 16, <= 256; multiple of 32 when B is MN-major)
  int net;                    // 0 = discriminator, 1 = generator (which lr_t k_dw_adam_tc uses)
  int ws_stride;              // split-K (large-batch dW): floats between the partial products of two contraction slices
  float* ws;                  // ... and their workspace, laid out like C; k_splitk_reduce sums the slices in a fixed order
  int esz;                    // operand element size: 4 (or 0) = fp32 read as tf32, 2 = fp16 copies (kind::f16, fp32 accumulation)
  int head;                   // HEAD_*: reduction fused into this GEMM's epilogue
  int stats_stride;           // floats between the statistics blocks of two batches of the epoch
  const void* hd;             // the fold's LossDesc (HEAD_DISC / HEAD_FM) or BnDesc (HEAD_BN)
  float* stats;               // the fold's block of 4 step statistics at batch 0
};

#define TC_KBLK 32            // contraction elements per stage (one 128-byte swizzle row of fp32)
#define TC_SPIN_LIMIT (1ll << 31)   // cycles; a stuck barrier traps instead of hanging the GPU

#ifdef MRGAN_PHASE_TIMING
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define PT_MARK(i) do { pt[i] = gtimer(); } while (0)
#else
#define PT_MARK(i) do { } while (0)
#endif

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%1], %0;" ::"r"(count), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%1], %0;" ::"r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > TC_SPIN_LIMIT) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void prefetch_map(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor (version 1).  lbo/sbo in bytes.
//   K-major operand : layout 2 = SWIZZLE_128B (16-byte chunks XOR row&7; TMA SWIZZLE_128B), sbo = 8 rows = 1024 B
//   MN-major operand: 32-bit types only support layout 1 = SWIZZLE_128B_BASE32B (32-byte chunks XOR k-row&3;
//                     TMA SWIZZLE_128B_ATOM_32B): 4 k-rows of 128 B per atom -> sbo = 512 B, lbo = next 32-element MN block
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float v[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Asynchronous TMEM loads: issue any number, wait once, then pass each destination array through tmem_fence16 -- an empty
// volatile asm that "modifies" the registers, so no use of them can be scheduled ahead of the wait.
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence16(uint32_t (&r)[16]) {
  asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                    "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]) :: "memory");
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float v[8]) {
  uint32_t r[8];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float v[4]) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float v[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3]))
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float v[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

}  // namespace tc


// ---- epilogue row processors: one 16-row chunk of one feature (= thread).  Everything that is uniform over the launch
// (activation, which outputs exist, operand formats) is a template parameter, so a row costs ~10 instructions instead
// of ~60 of branchy code; the chunk loops dispatch once per chunk.  Pointers walk down the rows by the pitch.
// Global stores of the epilogues: plain st.global (the output pointers are never in another state space; a generic ST would
// carry the state-space check) of one element per row, addressed as base + j * pitch so that no pointer chain links the rows.
__device__ __forceinline__ void stg_f32(float* p, float v) { asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }
__device__ __forceinline__ void stg_h16(__half* p, __half v) { asm volatile("st.global.b16 [%0], %1;" ::"l"(p), "h"(__half_as_ushort(v)) : "memory"); }

// FULL: all 16 rows of the chunk exist (every chunk but the last of a tile) -- no per-row predicate at all.  The branches
// on c_op / c2_op are uniform over the launch and sit outside the row loops, so a row is ~8 straight-line instructions.
template <bool F16, int ACT, bool HAS_C, bool HAS_C2, bool FULL>
__device__ __forceinline__ void fwd_rows(const uint32_t (&va)[16], const float (&nz)[16], int nrows, float* pC, __half* hC, int ldc,
                                         bool c_op, float* pC2, __half* hC2, int ldc2, bool c2_op, float sigma, float alpha, bool mul) {
  float x[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    float v = __uint_as_float(va[j]);
    if (!F16) v *= TF32_TRUNC_DEBIAS;
    if (ACT == ACT_RELU) v = fmaxf(v, 0.f);
    else if (ACT == ACT_SOFTPLUS) v = softplus_fast(v);
    else if (ACT == ACT_LEAKY) v = v > 0.f ? v : alpha * v;
    x[j] = v;
  }
  if (HAS_C) {                  // clean activation: kept in fp32 (act' of the backward pass, feature matching, logits) ...
    if (!F16 && c_op) {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_f32(pC + (uint32_t)(j * ldc), rna_tf32(x[j]));
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_f32(pC + (uint32_t)(j * ldc), x[j]);
    }
    if (F16 && c_op) {          // ... plus its 16-bit operand copy where a GEMM reads it
#pragma unroll
      for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_h16(hC + (uint32_t)(j * ldc), __float2half_rn(x[j]));
    }
  }
  if (HAS_C2) {                 // noisy activation: only ever a GEMM operand
    float y[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) y[j] = mul ? x[j] * nz[j] : fmaf(sigma, nz[j], x[j]);      // Dropout keep factor / GaussianNoise
    if (F16 && c2_op) {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_h16(hC2 + (uint32_t)(j * ldc2), __float2half_rn(y[j]));
    } else if (!F16 && c2_op) {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_f32(pC2 + (uint32_t)(j * ldc2), rna_tf32(y[j]));
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_f32(pC2 + (uint32_t)(j * ldc2), y[j]);
    }
  }
}

// ACT_RELU / ACT_LEAKY: av is the layer's clean output h (slope 1 where h > 0, else alpha; alpha = 0 for ReLU) -- or, when a
// Dropout layer follows the activation (dinv = 1 / (1 - rate)), its DROPPED output a = f h: the element was dropped iff
// a == 0, and a kept element has the sign of h, so one array carries both derivatives.
template <bool F16, int ACT, bool FULL>
__device__ __forceinline__ void dx_rows(const uint32_t (&va)[16], const float (&av)[16], int nrows, float* pC, __half* hC, int ldc, bool op_only,
                                        float alpha, float dinv, bool drop) {
  float x[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    float v = __uint_as_float(va[j]);
    if (!F16) v *= TF32_TRUNC_DEBIAS;
    if (ACT == ACT_RELU || ACT == ACT_LEAKY) {
      float m = (av[j] > 0.f ? 1.0f : (ACT == ACT_LEAKY ? alpha : 0.f)) * dinv;
      if (drop && av[j] == 0.f) m = 0.f;
      v *= m;
    } else if (ACT == ACT_SOFTPLUS) v *= 1.0f - __expf(-av[j]);
    x[j] = v;
  }
  if (F16 && op_only) {         // operand only: 16-bit copy, loss-scaled like the accumulator
#pragma unroll
    for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_h16(hC + (uint32_t)(j * ldc), grad_to_half(x[j]));
  } else if (!F16 && op_only) {
#pragma unroll
    for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_f32(pC + (uint32_t)(j * ldc), rna_tf32(x[j]));
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) if (FULL || j < nrows) stg_f32(pC + (uint32_t)(j * ldc), x[j]);
  }
}


// ---- fused heads: a second pass over the finished accumulator (TMEM reads are cheap) by the epilogue warps -----------
// One 16-row chunk of this thread's feature from TMEM, as the activation the forward epilogue stored.
template <bool F16, int ACT>
__device__ __forceinline__ void head_chunk(uint32_t taddr, float (&x)[16], float alpha = 0.f) {
  tc::tmem_ld16(taddr, x);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    if (!F16) x[j] *= TF32_TRUNC_DEBIAS;
    if (ACT == ACT_RELU) x[j] = fmaxf(x[j], 0.f);
    else if (ACT == ACT_SOFTPLUS) x[j] = softplus_fast(x[j]);
    else if (ACT == ACT_LEAKY) x[j] = x[j] > 0.f ? x[j] : alpha * x[j];
  }
}

// HEAD_DISC: Salimans-style supervised + unsupervised losses on the stacked rows [labeled | unlabeled | fake]
// (mr_gan.py:146-149,161) and the closed-form logit gradients (SURVEY.md 3.2).  The K logits of a row sit in lanes 0..K-1
// of the quadrant-0 warps; they are transposed through shared memory (the operand stages are free once the accumulator
// is complete) so that one THREAD handles one row, all epilogue warps in parallel.  Per-warp partial sums of (loss_lab,
// loss_unl, errors) go to part[3 * warp]; the caller adds them in warp order.
template <bool F16, int EPW>
__device__ __forceinline__ void head_disc(uint32_t trow, int cbeg, int ncols, int nall, int lane_base, int lane, int ewarp,
                                          const LossDesc& L, const AdamHyper& hp, const OperandMode& om, float* sl, float* part) {
  const int K = hp.n_classes, B = hp.dp_bloc;
  const float Bg = (float)hp.dp_bg;
  if (lane_base == 0) {
    for (int c0 = cbeg; c0 < ncols; c0 += 16) {
      float v[16];
      head_chunk<F16, ACT_NONE>(trow + (uint32_t)c0, v);
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (lane < K && c0 + j < ncols) sl[(c0 + j) * K + lane] = v[j];
    }
  }
  asm volatile("bar.sync 1, %0;" ::"r"(32 * EPW) : "memory");      // the epilogue warps only
  float s_lab = 0.f, s_unl = 0.f, s_err = 0.f;
  for (int r = ewarp * 32 + lane; r < nall; r += 32 * EPW) {
    const float* l = sl + r * K;
    float mx = l[0]; int am = 0;
    for (int k = 1; k < K; ++k) if (l[k] > mx) { mx = l[k]; am = k; }
    float se = 0.f;
    for (int k = 0; k < K; ++k) se += expf(l[k] - mx);
    const float lse = mx + logf(se), inv = 1.0f / se;
    float* dl = L.dlogits + (size_t)r * L.ld;
    if (r < B) {
      const int y = L.labels[r];
      s_lab += lse - l[y];
      s_err += (am != y) ? 1.f : 0.f;
      for (int k = 0; k < K; ++k) put_grad_operand(dl + k, (expf(l[k] - mx) * inv - (k == y ? 1.f : 0.f)) / Bg, om);
    } else {
      const float sp = softplusf(lse), sg = 1.0f / (1.0f + expf(-lse));
      float coef;
      if (r < 2 * B) { s_unl += 0.5f * (sp - lse); coef = 0.5f * (sg - 1.0f); }
      else           { s_unl += 0.5f * sp;         coef = 0.5f * sg; }
      coef *= hp.w_unl / Bg;
      for (int k = 0; k < K; ++k) put_grad_operand(dl + k, coef * expf(l[k] - mx) * inv, om);
    }
  }
  s_lab = warp_sum(s_lab); s_unl = warp_sum(s_unl); s_err = warp_sum(s_err);
  if (lane == 0) { part[3 * ewarp] = s_lab; part[3 * ewarp + 1] = s_unl; part[3 * ewarp + 2] = s_err; }
}

// HEAD_FM: rows [0,B) = fake, [B,2B) = real post-ReLU activations of D layer 5; this thread's feature f (MT = 2: the warp
// group owns all rows of its sub-tile).  Writes the warp's partial of sum_f diff_f^2 to *red and dZ5 (already multiplied by
// ReLU') for the fake rows (mr_gan.py:152-154).
template <bool F16, bool VAR>
__device__ __forceinline__ void head_fm(uint32_t trow, int ncols, int f, bool f_ok, int lane, const LossDesc& L, const AdamHyper& hp,
                                        const OperandMode& om, float* red) {
  constexpr int HACT = VAR ? ACT_LEAKY : ACT_RELU;      // alpha = 0 in the VAR kernels reproduces ReLU
  const int B = hp.dp_bloc;
  float mg = 0.f, mr = 0.f;
  for (int c0 = 0; c0 < ncols; c0 += 16) {
    float x[16];
    head_chunk<F16, HACT>(trow + (uint32_t)c0, x, hp.alpha);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int r = c0 + j;
      if (r < B) mg += x[j]; else if (r < ncols) mr += x[j];
    }
  }
  const float diff = (mg - mr) / B;
  const float part = warp_sum(f_ok ? diff * diff : 0.f);
  if (lane == 0) *red = part;
  float g = 2.0f * diff / ((float)L.Wmid * B);
  if (!F16) g = rna_tf32(g);
  for (int c0 = 0; c0 < B; c0 += 16) {
    float x[16];
    head_chunk<F16, HACT>(trow + (uint32_t)c0, x, hp.alpha);
    if (!f_ok) continue;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int r = c0 + j;
      if (r < B) put_grad_operand(L.dmid + (size_t)r * L.lddmid + f, x[j] > 0.f ? g : hp.alpha * g, om);
    }
  }
}

// HEAD_BN: BatchNormalization(epsilon) of G layer 1's softplus output in training phase (biased batch variance,
// mr_gan.py:112).  Statistics over ALL nall rows of this thread's feature (with one sub-tile per CTA both warp groups
// compute them, redundantly) in one pass of shifted sums (shift = the first row's value, which keeps E[d^2] - E[d]^2 well
// conditioned); xhat, 1/std and the GEMM operand u = gamma xhat + beta are written for rows [cbeg, ncols).
template <bool F16>
__device__ __forceinline__ void head_bn(uint32_t trow, int cbeg, int ncols, int nall, int f, bool f_ok, const BnDesc& Bd,
                                        const AdamHyper& hp, const OperandMode& om) {
  float s = 0.f, q = 0.f, x0 = 0.f;
  for (int c0 = 0; c0 < nall; c0 += 16) {
    float x[16];
    head_chunk<F16, ACT_SOFTPLUS>(trow + (uint32_t)c0, x);
    if (c0 == 0) x0 = x[0];
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c0 + j < nall) { const float d = x[j] - x0; s += d; q = fmaf(d, d, q); }
  }
  const float md = s / nall, mu = x0 + md;
  const float istd = rsqrtf(fmaxf(q / nall - md * md, 0.f) + hp.bn_eps);
  float ga = 0.f, be = 0.f;
  if (f_ok) { if (cbeg == 0) Bd.istd[f] = istd; ga = Bd.gamma[f]; be = Bd.beta[f]; }
  for (int c0 = cbeg; c0 < ncols; c0 += 16) {
    float x[16];
    head_chunk<F16, ACT_SOFTPLUS>(trow + (uint32_t)c0, x);
    if (!f_ok) continue;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int r = c0 + j;
      if (r >= ncols) break;
      const float xh = (x[j] - mu) * istd;
      Bd.xhat[(size_t)r * Bd.ld + f] = xh;
      put_operand(Bd.u + (size_t)r * Bd.ldu + f, fmaf(ga, xh, be), om);
    }
  }
}

// A_MN / B_MN: operand is MN-major (its MMA M/N dimension is the memory-contiguous one).  The pair also selects the role:
//   A_MN && !B_MN  forward   (EPI_FWD)      !A_MN && !B_MN  dX (EPI_DX)      A_MN && B_MN  dW (EPI_STORE)
// STAGES: depth of the TMA->MMA ring; TMEM_COLS: TMEM columns allocated (power of 2 >= MT x bn);
// MINB: CTAs per SM the register allocation must allow; EPW: epilogue warps (4 or 8; with 8 and MT == 1 the accumulator
// columns are split between two warp groups).
// MT: feature sub-tiles of 128 per CTA (1 or 2).  With MT = 2 the CTA computes 256 features against ONE copy of the
// batch-side operand tile (two accumulators in TMEM, 2 x 4 MMAs per stage), which cuts the activation bytes every SM has to
// ingest -- the forward / dX mainloops run at the L2->SM ingest limit (measured 0.9 - 1.0 us per 52 KB stage and SM) -- and
// each warp group of the epilogue owns one sub-tile.  MT = 2 requires EPW = 8 and TMEM_COLS = 512.
// F16: operands are 16-bit copies (kind::f16: fp16 weights / activations / loss-scaled gradients): a 128-byte swizzle row
// holds 64 contraction elements, an MMA covers K = 16, an MN-major box is 64 elements x 64 contraction rows (plain 128B
// swizzle, UMMA layout 2, SBO 1024 B, LBO 8192 B); otherwise fp32 operands read as tf32 (32 elements per row, K = 8 per
// MMA, MN-major boxes of 32 x 32 with the 32-byte-atom swizzle, UMMA layout 1, SBO 512 B, LBO 4096 B).  Compile-time,
// so every descriptor constant folds and the single-thread producer / issuer loops unroll.
// VAR: the LeakyReLU / Dropout variants of the discriminator (others/wganlpctsemi.py:166-179) are compiled in.  A separate
// instantiation, because carrying them in the reference configuration's epilogues measured 2.3 % of the whole step.
template <bool A_MN, bool B_MN, int STAGES, int TMEM_COLS, int MINB, int EPW, int MT, bool F16, bool VAR>
__global__ void __launch_bounds__(64 + 32 * EPW, MINB)
k_gemm_tc(const TcOp* __restrict__ ops, FoldState* __restrict__ folds, int rows_override, AdamHyper hp, OperandMode om) {
  using namespace tc;
#ifdef MRGAN_PHASE_TIMING
  const unsigned long long pt_t0 = gtimer();
#endif
  constexpr int KBLK = F16 ? 64 : 32;                 // contraction elements per stage (one 128-byte row)
  constexpr uint32_t MN_BOX = F16 ? 8192u : 4096u;    // bytes of one MN-major box (KBLK elements x KBLK contraction rows)
  // dW (B_MN) kernels take the number of contraction slices in `rows_override`: blockIdx.z = fold * ksplit + slice, each
  // slice stores its partial product to op.ws (deterministic split-K: a fold's dW of the narrow layers is one or two
  // tiles, which would leave a large-batch contraction of thousands of rows on one or two SMs)
  const int ksplit = (B_MN && rows_override > 1) ? rows_override : 1;
  const int kslice = (int)blockIdx.z % ksplit;
  const TcOp& op = ops[blockIdx.z / ksplit];
  const int ME = op.ME, KE = op.KE, bn = op.bn;
  int NE = op.NE;
  if (rows_override > 0 && !B_MN) NE = rows_override;      // fewer batch rows (G step)
  const int m0 = blockIdx.x * 128 * MT, n0 = blockIdx.y * bn;
  if (m0 >= ME || n0 >= NE) return;                         // uniform per CTA: nothing allocated yet

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t a_bytes = MT * 128 * 128, b_bytes = (uint32_t)bn * 128, stage_bytes = a_bytes + b_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * stage_bytes);
  uint64_t* full = bars;                    // [STAGES]
  uint64_t* empty = bars + STAGES;          // [STAGES]
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 1);
  float* const red = reinterpret_cast<float*>(bars + 24);    // 16 floats of head scratch at the end of the 256-byte barrier block
#ifdef MRGAN_PHASE_TIMING
  unsigned long long* pt = reinterpret_cast<unsigned long long*>(bars + 16);     // inside the 256-byte slack after the barriers
  if (threadIdx.x == 0) pt[0] = pt_t0;
#endif

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb_all = (KE + KBLK - 1) / KBLK;
  const int kb_per = (nkb_all + ksplit - 1) / ksplit;
  const int kb0 = kslice * kb_per;                           // the host picks ksplit so that no slice is empty
  const int nkb = min(nkb_all, kb0 + kb_per) - kb0;

  if (warp == 0 && lane == 0) {
    prefetch_map(&op.mapA);
    prefetch_map(&op.mapB);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // TMEM: TMEM_COLS fp32 columns x 128 lanes for the accumulator tile
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"((uint32_t)TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = *tmem_holder;
  if (threadIdx.x == 0) PT_MARK(1);

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_expect_tx(&full[s], stage_bytes);
        uint8_t* sa = smem + (size_t)s * stage_bytes;
        uint8_t* sb = sa + a_bytes;
        const int k0 = (kb0 + kb) * KBLK;
        if (A_MN) {
#pragma unroll
          for (int b = 0; b < (128 / KBLK) * MT; ++b) tma_load_2d(&op.mapA, &full[s], sa + b * MN_BOX, m0 + KBLK * b, k0);
        } else {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) tma_load_2d(&op.mapA, &full[s], sa + mt * 16384, k0, m0 + 128 * mt);
        }
        if (B_MN) {
          for (int b = 0; b < bn / KBLK; ++b) tma_load_2d(&op.mapB, &full[s], sb + b * MN_BOX, n0 + KBLK * b, k0);
        } else {
          tma_load_2d(&op.mapB, &full[s], sb, k0, n0);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      // instruction descriptor: D format f32 (1 << 4); operand formats (bits 7-9 / 10-12): 0 = f16, 2 = tf32; majors; N >> 3; M >> 4
      constexpr uint32_t fmt = F16 ? 0u : 2u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                             ((uint32_t)(bn >> 3) << 17) | ((128u >> 4) << 24);
      constexpr uint32_t mn_lbo = MN_BOX, mn_sbo = F16 ? 1024u : 512u, mn_lay = F16 ? 2u : 1u, mn_step = F16 ? 2048u : 1024u;
      constexpr uint32_t lboA = A_MN ? mn_lbo : 16u, lboB = B_MN ? mn_lbo : 16u;
      constexpr uint32_t sboA = A_MN ? mn_sbo : 1024u, sboB = B_MN ? mn_sbo : 1024u;
      constexpr uint32_t layA = A_MN ? mn_lay : 2u, layB = B_MN ? mn_lay : 2u;
      constexpr uint32_t stepA = A_MN ? mn_step : 32u, stepB = B_MN ? mn_step : 32u;   // bytes per MMA (8 tf32 / 16 f16 contraction elements)
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
        mbar_wait(&full[s], ph);
        if (kb == 0) PT_MARK(2);
        fence_after();
        const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes), sb = sa + a_bytes;
#pragma unroll
        for (int k = 0; k < 4; ++k) {            // 4 MMAs per stage and sub-tile in both formats
          const uint64_t db = smem_desc(sb + k * stepB, lboB, sboB, layB);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {      // sub-tile mt: A block at +16 KB, accumulator at TMEM column 256 * mt
            const uint64_t da = smem_desc(sa + mt * 16384u + k * stepA, lboA, sboA, layA);
            if (F16) mma_f16(tmem_base + 256u * mt, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            else mma_tf32(tmem_base + 256u * mt, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
        }
        mma_commit(&empty[s]);            // frees the smem stage when these MMAs retire
      }
      mma_commit(tmem_full);              // accumulator complete
      PT_MARK(3);
    }
  } else {
    // ===================== epilogue (EPW warps; a warp may only touch TMEM lanes 32*(warp%4)..+31) =====================
    const int lane_base = 32 * (warp & 3);
    const int wg = (warp - 2) >> 2;                       // epilogue warp group (0 or 1 when EPW == 8)
    const int sub = (MT == 2) ? wg : 0;                   // MT == 2: one feature sub-tile per warp group
    const int chalf = (EPW == 8 && MT == 1) ? (((min(bn, NE - n0) + 1) / 2 + 15) & ~15) : bn;   // columns per warp group
    const int cbeg = (EPW == 8 && MT == 1) ? wg * chalf : 0;
    const int f = m0 + 128 * sub + lane_base + lane;      // this thread's feature index (MMA-M)
    const bool f_ok = f < ME;
    const GemmDesc g = op.g;             // by value: descriptor fields must not be re-read from HBM around every store
    constexpr float debias = F16 ? 1.0f : TF32_TRUNC_DEBIAS;   // fp16 operand copies are rounded to nearest: nothing to remove
    const int ncols = min(min(bn, NE - n0), cbeg + chalf);      // this warp's column range is [cbeg, ncols)
    const uint32_t trow = tmem_base + 256u * sub + ((uint32_t)lane_base << 16);
    // TMEM columns the accumulators leave free: scratch of this warp group (sub-tile s owns [256 s + bn, 256 s + 256); with
    // one sub-tile the warp groups share [bn, TMEM_COLS)), in whole 16-column chunks
    int fbeg, flen;
    if (MT == 2) { fbeg = 256 * sub + bn; flen = (256 - bn) & ~15; }
    else { flen = ((TMEM_COLS - bn) / (EPW == 8 ? 2 : 1)) & ~15; fbeg = bn + wg * flen; }
    const uint32_t tfree = tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)fbeg;
    const int nchunks = (ncols - cbeg + 15) >> 4;               // 16-row chunks of this warp's range (<= 0: nothing to do)
    const int npark = max(min(flen >> 4, nchunks), 0);          // chunks whose noise / h values fit the free columns

    if constexpr (B_MN) {
      // ------------------------------------------------------------------ dW: EPI_STORE into the flat gradient buffer
      // (large-batch / data-parallel mode: Adam follows on the all-reduced gradient; the reference batch uses k_dw_adam_tc)
      mbar_wait(tmem_full, 0);
      fence_after();
      float* const dst = ksplit > 1 ? op.ws + (size_t)kslice * op.ws_stride : g.C;
      for (int c0 = cbeg; c0 < ncols; c0 += 16) {
        float v[16];
        tmem_ld16(trow + (uint32_t)c0, v);                   // warp-collective: every lane takes part
        if (!f_ok) continue;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int k = n0 + c0 + j;
          if (k >= NE) break;
          dst[(size_t)k * g.ldc + f] = v[j];
        }
      }
    } else if constexpr (!A_MN) {
      // ------------------------------------------------------------------ dX: dZ_prev[r, f] = acc * act'(h_prev[r, f])
      // The h values do not depend on the accumulator: whole 16-row chunks of them are loaded while the mainloop runs and
      // parked in the free TMEM columns; chunks that do not fit are register-prefetched one chunk ahead.  Per chunk the
      // accumulator and the parked values are fetched with two TMEM loads behind ONE wait.
      const bool has_act = g.act != ACT_NONE;
      // Dropout variant: aux is the layer's DROPPED output a (see dx_rows), which in f16 mode exists only as the fp16 copy
      const bool drop = VAR && hp.drop > 0.f && (g.act == ACT_RELU || g.act == ACT_LEAKY) && g.tid >= 1;
      const __half* const haux = (F16 && drop) ? om.hbase + (g.aux - om.fbase) : nullptr;
      auto fetch = [&](int c0, float (&av)[16]) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const size_t o = (size_t)(n0 + c0 + j) * g.ldaux + f;
          av[j] = (f_ok && has_act && c0 + j < ncols) ? (haux ? __half2float(haux[o]) : __ldg(g.aux + o)) : 1.0f;
        }
      };
      float avA[16], avB[16];
      const int npk = has_act ? npark : 0;
      if (npk > 0) {
        fetch(cbeg, avA);
        for (int k = 0; k < npk; k += 2) {
          if (k + 1 < npk) fetch(cbeg + 16 * (k + 1), avB);
          tmem_st16(tfree + 16u * (uint32_t)k, avA);
          if (k + 1 < npk) {
            if (k + 2 < npk) fetch(cbeg + 16 * (k + 2), avA);
            tmem_st16(tfree + 16u * (uint32_t)(k + 1), avB);
          }
        }
        tmem_wait_st();
      }
      if (has_act && npk < nchunks) fetch(cbeg + 16 * npk, avA);
      mbar_wait(tmem_full, 0);
      fence_after();
      __half* const hC = F16 ? om.hbase + (g.C - om.fbase) : nullptr;
      const bool op_only = (g.rnd & 1) != 0;                      // the result is only ever a GEMM operand
      for (int ch = 0; ch < nchunks; ++ch) {
        const int c0 = cbeg + 16 * ch;
        uint32_t va[16], vh[16];
        tmem_ld16_issue(trow + (uint32_t)c0, va);
        if (ch < npk) tmem_ld16_issue(tfree + 16u * (uint32_t)ch, vh);
        tmem_wait_ld();
        tmem_fence16(va);
        float av[16];
        if (ch < npk) {
          tmem_fence16(vh);
#pragma unroll
          for (int j = 0; j < 16; ++j) av[j] = __uint_as_float(vh[j]);
        } else if (has_act) {
          const bool odd = ((ch - npk) & 1) != 0;
#pragma unroll
          for (int j = 0; j < 16; ++j) av[j] = odd ? avB[j] : avA[j];
          if (ch + 1 < nchunks) { if (odd) fetch(c0 + 16, avA); else fetch(c0 + 16, avB); }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) av[j] = 1.0f;
        }
        if (!f_ok) continue;
        const size_t o0 = (size_t)(n0 + c0) * g.ldc + f;
        const int nrows = ncols - c0;
        float* const pC = g.C + o0;
        __half* const phC = F16 ? hC + o0 : nullptr;
        const float dinv = drop ? hp.drop_inv : 1.0f;
#define DX_ACT(FULL)                                                                                                        \
        do {                                                                                                                    \
          if (g.act == ACT_RELU) dx_rows<F16, ACT_RELU, FULL>(va, av, nrows, pC, phC, g.ldc, op_only, 0.f, dinv, drop);         \
          else if (VAR && g.act == ACT_LEAKY) dx_rows<F16, ACT_LEAKY, FULL>(va, av, nrows, pC, phC, g.ldc, op_only, hp.alpha, dinv, drop); \
          else if (g.act == ACT_SOFTPLUS) dx_rows<F16, ACT_SOFTPLUS, FULL>(va, av, nrows, pC, phC, g.ldc, op_only, 0.f, 1.0f, false);      \
          else dx_rows<F16, ACT_NONE, FULL>(va, av, nrows, pC, phC, g.ldc, op_only, 0.f, 1.0f, false);                          \
        } while (0)
        if (nrows >= 16) DX_ACT(true); else DX_ACT(false);
#undef DX_ACT
      }
    } else {
      // ------------------------------------------------------------------ forward: act, optional clean copy, noisy copy
      // GaussianNoise of the next layer's input (C2): the draws do not depend on the accumulator, and the epilogue warps are
      // idle while the TMA / MMA warps run the mainloop -- so they draw now and park whole 16-row chunks in the free TMEM
      // columns.  Chunks that do not fit are drawn in the epilogue BETWEEN issuing the accumulator's TMEM load and waiting
      // for it, so the Philox rounds hide the load latency; per chunk there is one wait for both TMEM loads.
      // Dropout variant (hp.drop > 0): the transforms in front of D's hidden layers 2..5 (stream ids 1..4) are Dropout(rate)
      // instead of GaussianNoise: the parked / drawn values are keep factors and combine by multiplication
      const bool mul = VAR && hp.drop > 0.f && g.C2 != nullptr && g.tid >= 1;
      const float ddrop = mul ? hp.drop : 0.f;
      const bool noisy = g.C2 != nullptr && (g.sigma != 0.f || mul);
      uint32_t key0 = 0, key1 = 0, step = 0;
      if (noisy) { const FoldState& fs = folds[g.fold]; key0 = fs.key0; key1 = fs.key1; step = (uint32_t)fs.rng_step; }
      // 4-row noise groups must not straddle row-section or rank boundaries (oracle/philox.py): otherwise per-element draws
      const bool grp = ((g.row0 + n0 + cbeg) & 3) == 0 && (hp.dp_bg == hp.dp_bloc || (hp.dp_bloc & 3) == 0);
      const bool dp = hp.dp_bg != hp.dp_bloc;
      const int dprank = hp.dp_rank < 0 ? g.fold : hp.dp_rank;      // virtual-rank mode: the fold is the rank
      auto draw16 = [&](int c0, float (&nz)[16]) {
        const int r0 = g.row0 + n0 + c0;
        if (grp && !dp) {
          // the common case: four independent Philox chains, inlined so the compiler interleaves them (the epilogue warps
          // are latency-bound here: 2 warps per scheduler)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (VAR) noise_or_drop4(key0, key1, (uint32_t)(r0 + 4 * q) >> 2, (uint32_t)f, step, (uint32_t)g.tid, ddrop, hp.drop_inv, &nz[4 * q]);
            else normal4(key0, key1, (uint32_t)(r0 + 4 * q) >> 2, (uint32_t)f, step, (uint32_t)g.tid, &nz[4 * q]);
          }
        } else if (grp) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 n4 = noise4_call(key0, key1, r0 + 4 * q, (uint32_t)f, step, (uint32_t)g.tid, hp.dp_bloc, hp.dp_bg, dprank, ddrop, hp.drop_inv);
            nz[4 * q] = n4.x; nz[4 * q + 1] = n4.y; nz[4 * q + 2] = n4.z; nz[4 * q + 3] = n4.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            nz[j] = noise1_call(key0, key1, r0 + j, (uint32_t)f, step, (uint32_t)g.tid, hp.dp_bloc, hp.dp_bg, dprank, ddrop, hp.drop_inv);
        }
      };
      const int npk = (noisy && grp) ? npark : 0;
      for (int ch = 0; ch < npk; ++ch) {
        float nz[16];
        draw16(cbeg + 16 * ch, nz);
        tmem_st16(tfree + 16u * (uint32_t)ch, nz);
      }
      if (npk > 0) tmem_wait_st();
      if (warp == 2 && lane == 0) PT_MARK(4);
      mbar_wait(tmem_full, 0);
      if (warp == 2 && lane == 0) PT_MARK(5);
      fence_after();
      __half* const hC = (F16 && g.C) ? om.hbase + (g.C - om.fbase) : nullptr;
      __half* const hC2 = (F16 && g.C2) ? om.hbase + (g.C2 - om.fbase) : nullptr;
      const bool c_op = (g.rnd & 1) != 0, c2_op = (g.rnd & 2) != 0;   // C / C2 feed a tensor-core GEMM as operands
#ifdef MRGAN_PHASE_TIMING
      unsigned long long tch[24];
#endif
      // The second warp group walks its chunks backwards: the two warps that share a scheduler (one of each group) then work on
      // a parked chunk (store-bound) and a drawn chunk (ALU-bound) at the same time instead of both on the same kind.
      for (int it = 0; it < nchunks; ++it) {
        const int ch = (wg & 1) ? nchunks - 1 - it : it;
        const int c0 = cbeg + 16 * ch;
        uint32_t va[16], vn[16];
        float nz[16];
#ifdef MRGAN_PHASE_TIMING
        if (ch < 12) tch[2 * ch] = gtimer();
#endif
        tmem_ld16_issue(trow + (uint32_t)c0, va);
        if (ch < npk) tmem_ld16_issue(tfree + 16u * (uint32_t)ch, vn);
        else if (noisy) draw16(c0, nz);                        // overlaps the accumulator load
        tmem_wait_ld();
#ifdef MRGAN_PHASE_TIMING
        if (ch < 12) tch[2 * ch + 1] = gtimer();
#endif
        tmem_fence16(va);
        if (ch < npk) {
          tmem_fence16(vn);
#pragma unroll
          for (int j = 0; j < 16; ++j) nz[j] = __uint_as_float(vn[j]);
        }
        if (!f_ok) continue;
        const size_t o0 = (size_t)(n0 + c0) * g.ldc + f, o20 = (size_t)(n0 + c0) * g.ldc2 + f;
        const int nrows = ncols - c0;
        float* const pC = g.C ? g.C + o0 : nullptr;
        float* const pC2 = g.C2 ? g.C2 + o20 : nullptr;
        __half* const phC = hC ? hC + o0 : nullptr;
        __half* const phC2 = hC2 ? hC2 + o20 : nullptr;
        if (!noisy) {
#pragma unroll
          for (int j = 0; j < 16; ++j) nz[j] = 0.f;
        }
#define FWD_ROWS(ACT, HC, HC2, FULL) \
        fwd_rows<F16, ACT, HC, HC2, FULL>(va, nz, nrows, pC, phC, g.ldc, c_op, pC2, phC2, g.ldc2, c2_op, g.sigma, hp.alpha, VAR && mul)
#define FWD_ACT(HC, HC2, FULL)                                                     \
        do {                                                                       \
          if (g.act == ACT_RELU) FWD_ROWS(ACT_RELU, HC, HC2, FULL);                \
          else if (g.act == ACT_SOFTPLUS) FWD_ROWS(ACT_SOFTPLUS, HC, HC2, FULL);   \
          else if (VAR && g.act == ACT_LEAKY) FWD_ROWS(ACT_LEAKY, HC, HC2, FULL);  \
          else FWD_ROWS(ACT_NONE, HC, HC2, FULL);                                  \
        } while (0)
#define FWD_OUT(FULL)                                                              \
        do {                                                                       \
          if (g.C && g.C2) FWD_ACT(true, true, FULL);                              \
          else if (g.C) FWD_ACT(true, false, FULL);                                \
          else if (g.C2) FWD_ACT(false, true, FULL);                               \
        } while (0)
        if (nrows >= 16) FWD_OUT(true); else FWD_OUT(false);
#undef FWD_OUT
#undef FWD_ACT
#undef FWD_ROWS
      }
#ifdef MRGAN_PHASE_TIMING
      if (warp == 2 && lane == 0 && blockIdx.x == 0 && blockIdx.z == 0 && nchunks >= 10) {
        const unsigned long long te2 = gtimer();
        const unsigned long long b = pt[0];
        printf("PTCH npk=%d: %llu+%llu %llu+%llu %llu+%llu %llu+%llu %llu+%llu %llu+%llu %llu+%llu %llu+%llu %llu+%llu %llu+%llu end=%llu\n", npk,
               tch[0] - b, tch[1] - tch[0], tch[2] - b, tch[3] - tch[2], tch[4] - b, tch[5] - tch[4], tch[6] - b, tch[7] - tch[6], tch[8] - b, tch[9] - tch[8],
               tch[10] - b, tch[11] - tch[10], tch[12] - b, tch[13] - tch[12], tch[14] - b, tch[15] - tch[14], tch[16] - b, tch[17] - tch[16],
               tch[18] - b, tch[19] - tch[18], te2 - b);
      }
#endif
      // ---- reductions fused into this GEMM (the host selects them only for single-tile batches outside the DP mode) ----
      if (op.head == HEAD_DISC) {       // scratch: operand stage 0 (every MMA has retired); partial sums behind the logits
        float* const sl = reinterpret_cast<float*>(smem);
        head_disc<F16, EPW>(trow, cbeg, ncols, min(bn, NE - n0), lane_base, lane, warp - 2, *static_cast<const LossDesc*>(op.hd), hp, om,
                            sl, sl + 8192);
      } else if (op.head == HEAD_FM) {  // MT == 2 (host): this warp group owns its sub-tile's features and all rows
        head_fm<F16, VAR>(trow, ncols, f, f_ok, lane, *static_cast<const LossDesc*>(op.hd), hp, om, red + (warp - 2));
      } else if (op.head == HEAD_BN) {
        head_bn<F16>(trow, cbeg, ncols, min(bn, NE - n0), f, f_ok, *static_cast<const BnDesc*>(op.hd), hp, om);
      }
    }
  }

  if (warp == 2 && lane == 0) PT_MARK(6);
  fence_before();
  __syncthreads();
  if (warp == 1) {
    fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
  }
  if (!B_MN && A_MN && threadIdx.x == 0 && (op.head == HEAD_DISC || op.head == HEAD_FM)) {
    // publish the step statistics (partials added in a fixed order); HEAD_DISC also advances the discriminator step's
    // K.update_add(iterations, 1) and noise step, since no k_adam launch follows it: nothing later in this step reads either
    float* const st = op.stats + (size_t)hp.t * op.stats_stride;
    if (op.head == HEAD_DISC) {
      const float Bg = (float)hp.dp_bg;
      const float* part = reinterpret_cast<const float*>(smem) + 8192;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      for (int w = 0; w < EPW; ++w) { a0 += part[3 * w]; a1 += part[3 * w + 1]; a2 += part[3 * w + 2]; }
      st[0] = a0 / Bg; st[1] = a1 / Bg; st[2] = a2 / Bg;
      FoldState& fs = folds[op.g.fold];
      if (hp.shared_t) fs.iterations += 1; else fs.it_net[0] += 1;
      fs.rng_step += 1;
    } else {
      float sum = 0.f;
      for (int w = 0; w < EPW; ++w) sum += red[w];
      st[3] = sum / static_cast<const LossDesc*>(op.hd)->Wmid;
    }
  }
#ifdef MRGAN_PHASE_TIMING
  if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0 && (blockIdx.z % 24) == 0) {
    const unsigned long long te = gtimer();
    printf("PT z=%d grid=(%d,%d,%d) nkb=%d t0=%llu setup=%llu first=%llu mma_issued=%llu noise=%llu acc=%llu epi=%llu end=%llu\n", (int)blockIdx.z,
           (int)gridDim.x, (int)gridDim.y, (int)gridDim.z, nkb, pt[0], pt[1] - pt[0], pt[2] - pt[0], pt[3] - pt[0], pt[4] - pt[0], pt[5] - pt[0], pt[6] - pt[0], te - pt[0]);
  }
#endif
}

// Sums the `ks` contraction slices of a split-K dW in slice order (bitwise reproducible) into the gradient tensor.
__global__ void __launch_bounds__(256) k_splitk_reduce(const TcOp* __restrict__ ops, int ks) {
  const TcOp& op = ops[blockIdx.y];
  const size_t n4 = (size_t)op.NE * op.g.ldc / 4, stride4 = (size_t)op.ws_stride / 4;
  const float4* __restrict__ ws = reinterpret_cast<const float4*>(op.ws);
  float4* __restrict__ out = reinterpret_cast<float4*>(op.g.C);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 a = ws[i];
    for (int s = 1; s < ks; ++s) {
      const float4 b = ws[(size_t)s * stride4 + i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    out[i] = a;
  }
}

// ====================================================================================================
// k_dw_adam_tc -- dW (+db) on tcgen05 with the Keras-2.0.9 Adam update fused in, optimizer state staged by TMA.
//
// grad(Waug_l)[k, n] = sum_r A[r, k] dZ[r, n]  as  D[n (128 lanes), k (128 columns)], then for the same tile
//   m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; W -= lr_t m / (sqrt(v) + eps)              (SURVEY.md 3.4, a8)
// W, m and v tiles never go through the LSU: one thread streams them HBM -> smem -> HBM in [KC rows x 128 cols]
// chunks with cp.async.bulk.tensor (full 128-byte lines, deep queues); the 4 epilogue warps combine each chunk
// with the matching 8 accumulator columns from TMEM in shared memory.  24 B per parameter of HBM traffic, which
// is the algorithmic minimum for Adam; the gradient never leaves the SM.  F16 (operand-copy mode): the operands are the
// 16-bit copies and every chunk also carries the fp16 copy of the UPDATED weights that the next forward / dX pass reads
// (written to smem by the epilogue, stored by TMA: +2 B per parameter).
//   smem: 2 operand stages x 16 KB + 3 chunk buffers x (3 x KC x 512 B [+ KC x 256 B]); 3 CTAs per SM.
// ====================================================================================================
struct alignas(64) TcAdamOp {
  CUtensorMap mapA, mapB;          // dZ[r, n] and A[r, k], both MN-major operands
  CUtensorMap mapP, mapM, mapV;    // Waug, m, v as [rows k, cols n], box = 128 cols x KC rows, no swizzle
  CUtensorMap mapH;                // fp16 copy of Waug, same geometry (F16 only)
  int ME, NE, KE;                  // out-features n, in-features(+1) k, contraction rows r
  int fold;
  int net;
  float ginv;                      // 1 / loss scale carried by the dZ operand (1 unless fp16 copies)
};

#define TCA_KC 8

namespace tc {
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"((uint64_t)map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
}  // namespace tc

// KROWS: contraction rows (batch rows) per operand stage, 32 fp16 / 16 fp32: 16 KB operand stages, which let THREE CTAs
// share an SM: a CTA spends its first microseconds on TMEM allocation, barrier set-up and the operand round trips while only
// its first chunk buffers are in flight -- with three co-resident CTAs two of them are always streaming.
template <bool F16, int KROWS> struct TcAdamCfg {
  static_assert(KROWS == (F16 ? 32 : 16), "operand stage geometry: 16 KB stages");
  static constexpr int STAGES = 2, KC = TCA_KC, NB = 3;
  static constexpr int MINB = 3;                                            // CTAs per SM
  static constexpr uint32_t MN_BOX = 128u * KROWS;                          // one MN-major box: 128 bytes (64 fp16 / 32 fp32) x KROWS rows
  static constexpr uint32_t STAGE_BYTES = (F16 ? 4 : 8) * MN_BOX;           // A + B operand tiles (128 features each)
  static constexpr uint32_t ARR_BYTES = KC * 128 * 4;                       // one array (W, m or v) of one chunk
  static constexpr uint32_t HALF_BYTES = F16 ? KC * 128 * 2 : 0;            // fp16 copy of the chunk's updated weights
  static constexpr uint32_t CHUNK_BYTES = 3 * ARR_BYTES + HALF_BYTES;
  static constexpr int NX = (STAGES * STAGE_BYTES) / CHUNK_BYTES;           // chunk buffers carved out of the operand stages later
  static constexpr int NBUF = NB + NX;
  static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + (size_t)NB * CHUNK_BYTES + 256;
};

template <bool F16, int KROWS>
__global__ void __launch_bounds__(192, (TcAdamCfg<F16, KROWS>::MINB))
k_dw_adam_tc(const TcAdamOp* __restrict__ ops, FoldState* __restrict__ folds, AdamHyper hp, int nfl, int op_stride) {
  // blockIdx.z = layer * nfl + fold: ONE launch may cover several layers of the step (their descriptors are op_stride apart);
  // the narrow layers' own grids are too small to keep HBM busy (60 % of peak against 89 % for the wide ones)
  using namespace tc;
  using Cfg = TcAdamCfg<F16, KROWS>;
  constexpr int STAGES = Cfg::STAGES, KC = Cfg::KC, NB = Cfg::NB, NBUF = Cfg::NBUF;
  constexpr uint32_t STAGE_BYTES = Cfg::STAGE_BYTES, ARR_BYTES = Cfg::ARR_BYTES, CHUNK_BYTES = Cfg::CHUNK_BYTES;
  constexpr int KBLK = KROWS;
  constexpr uint32_t MN_BOX = Cfg::MN_BOX;
  constexpr int MN_BOXES = F16 ? 2 : 4;                      // boxes per 128 features (64 fp16 / 32 fp32 elements wide)
  constexpr int MN_W = F16 ? 64 : 32;                        // elements per box row
  const TcAdamOp& op = ops[((int)blockIdx.z / nfl) * op_stride + ((int)blockIdx.z % nfl)];
  const int ME = op.ME, NE = op.NE, KE = op.KE;
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 128;     // n-feature tile (lanes), k-feature tile (columns)
  if (m0 >= ME || n0 >= NE) return;

  extern __shared__ __align__(1024) uint8_t smem_dyn[];
  uint8_t* smem = smem_dyn;
  if ((smem_u32(smem) & 1023u) != 0) __trap();                // swizzled TMA tiles need 1024-byte alignment
  uint8_t* cbuf = smem + STAGES * STAGE_BYTES;                // NB dedicated chunk buffers
  uint64_t* bars = reinterpret_cast<uint64_t*>(cbuf + NB * CHUNK_BYTES);
  uint64_t* full = bars;                       // [STAGES]   operands landed
  uint64_t* empty = bars + STAGES;             // [STAGES]   operands consumed
  uint64_t* tmem_full = bars + 2 * STAGES;     //            accumulator complete (2 waiters: epilogue, DMA thread)
  uint64_t* cfull = bars + 2 * STAGES + 1;     // [NBUF]     optimizer-state chunk landed
  uint64_t* cdone = cfull + NBUF;              // [NBUF]     chunk updated in smem (128 arrivals)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(cdone + NBUF);
  auto buf_ptr = [&](int b) -> uint8_t* { return b < NB ? cbuf + (size_t)b * CHUNK_BYTES : smem + (size_t)(b - NB) * CHUNK_BYTES; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (KE + KBLK - 1) / KBLK;
  const int ncols = min(128, NE - n0);
  const int nch = (ncols + KC - 1) / KC;

  if (warp == 0 && lane == 0) {
    prefetch_map(&op.mapA); prefetch_map(&op.mapB); prefetch_map(&op.mapP); prefetch_map(&op.mapM); prefetch_map(&op.mapV);
    if (F16) prefetch_map(&op.mapH);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    for (int b = 0; b < NBUF; ++b) { mbar_init(&cfull[b], 1); mbar_init(&cdone[b], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(128u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    if (lane == 0) {
      // ---- DMA thread: optimizer-state chunks first (they do not depend on the MMA), then the operands ----
      auto load_chunk = [&](int c) {
        const int b = c % NBUF;
        uint8_t* dst = buf_ptr(b);
        mbar_expect_tx(&cfull[b], 3 * ARR_BYTES);
        tma_load_2d(&op.mapP, &cfull[b], dst, m0, n0 + c * KC);
        tma_load_2d(&op.mapM, &cfull[b], dst + ARR_BYTES, m0, n0 + c * KC);
        tma_load_2d(&op.mapV, &cfull[b], dst + 2 * ARR_BYTES, m0, n0 + c * KC);
      };
      for (int c = 0; c < NB && c < nch; ++c) load_chunk(c);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_expect_tx(&full[s], STAGE_BYTES);
        uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
        uint8_t* sb = sa + STAGE_BYTES / 2;
        const int k0 = kb * KBLK;
#pragma unroll
        for (int b = 0; b < MN_BOXES; ++b) tma_load_2d(&op.mapA, &full[s], sa + b * MN_BOX, m0 + MN_W * b, k0);
#pragma unroll
        for (int b = 0; b < MN_BOXES; ++b) tma_load_2d(&op.mapB, &full[s], sb + b * MN_BOX, n0 + MN_W * b, k0);
      }
      // the MMAs have consumed every operand stage once the accumulator is complete: the operand region now takes
      // NX more chunks in flight
      mbar_wait(tmem_full, 0);
      for (int c = NB; c < NBUF && c < nch; ++c) load_chunk(c);
      // ---- write-back of updated chunks; a buffer is refilled one chunk late so that the store which is reading it has
      //      had a whole chunk period to drain (wait_group.read 1 instead of a full stall per chunk) ----
      for (int c = 0; c < nch; ++c) {
        const int b = c % NBUF;
        mbar_wait(&cdone[b], (uint32_t)(c / NBUF) & 1u);
        const uint8_t* src = buf_ptr(b);
        tma_store_2d(&op.mapP, src, m0, n0 + c * KC);
        tma_store_2d(&op.mapM, src + ARR_BYTES, m0, n0 + c * KC);
        tma_store_2d(&op.mapV, src + 2 * ARR_BYTES, m0, n0 + c * KC);
        if (F16) tma_store_2d(&op.mapH, src + 3 * ARR_BYTES, m0, n0 + c * KC);
        bulk_commit();
        if (c >= 1 && c - 1 + NBUF < nch) {
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          load_chunk(c - 1 + NBUF);
        }
      }
      bulk_wait_read0();
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t fmt = F16 ? 0u : 2u;
      constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
      constexpr uint32_t lbo = MN_BOX, sbo = F16 ? 1024u : 512u, lay = F16 ? 2u : 1u, kstep = F16 ? 2048u : 1024u;
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
        mbar_wait(&full[s], ph);
        fence_after();
        const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES), sb = sa + STAGE_BYTES / 2;
#pragma unroll
        for (int k = 0; k < KROWS / (F16 ? 16 : 8); ++k) {     // MMAs of K = 16 (f16) / 8 (tf32) contraction rows
          const uint64_t da = smem_desc(sa + k * kstep, lbo, sbo, lay), db = smem_desc(sb + k * kstep, lbo, sbo, lay);
          if (F16) mma_f16(tmem_base, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          else mma_tf32(tmem_base, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
        }
        mma_commit(&empty[s]);
      }
      mma_commit(tmem_full);
    }
  } else {
    // ---- epilogue: 4 warps, thread = output feature n (TMEM lane = smem column) ----
    const int lane_base = 32 * (warp & 3);
    const int nl = lane_base + lane;
    const uint32_t trow = tmem_base + ((uint32_t)lane_base << 16);
    const float lr_t = folds[op.fold].lr_t[op.net];
    const float b1 = hp.b1, b2 = hp.b2, c1 = 1.0f - hp.b1, c2 = 1.0f - hp.b2, eps = hp.eps;
    const float ginv = op.ginv;
    mbar_wait(tmem_full, 0);
    fence_after();
    for (int c = 0; c < nch; ++c) {
      const int b = c % NBUF;
      float* sP = reinterpret_cast<float*>(buf_ptr(b));
      float* sM = sP + KC * 128;
      float* sV = sM + KC * 128;
      __half* sH = reinterpret_cast<__half*>(sV + KC * 128);
      float g[KC];
      tmem_ld8(trow + (uint32_t)(c * KC), g);
      mbar_wait(&cfull[b], (uint32_t)(c / NBUF) & 1u);
#pragma unroll
      for (int j = 0; j < KC; ++j) {
        const int i = j * 128 + nl;
        const float gr = F16 ? g[j] * ginv : g[j];
        const float m = fmaf(b1, sM[i], c1 * gr), v = fmaf(b2, sV[i], c2 * gr * gr);
        sM[i] = m; sV[i] = v;
        const float w = sP[i] - lr_t * __fdividef(m, sqrtf(v) + eps);
        sP[i] = w;
        if (F16) sH[i] = __float2half_rn(w);       // operand copy for the next forward / dX (the TMA store clips it like the fp32 tile)
      }
      fence_proxy_async();              // generic-proxy writes -> visible to the bulk store
      mbar_arrive(&cdone[b]);
    }
  }

  fence_before();
  __syncthreads();
  if (warp == 1) {
    fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128u) : "memory");
  }
}
