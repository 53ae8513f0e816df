// common.cuh -- shared device structs, Philox4x32-10 noise stream, small helpers.
//
// Layout conventions (see DESIGN.md "Data layout in HBM"):
//  * every matrix is row-major fp32 with a pitch rounded up to 4 floats; pad
//    columns are zero at allocation and are NEVER written by any kernel;
//  * a Dense layer's kernel W[in,out] and bias b[out] (mr_gan.py:111-128) are
//    stored as ONE augmented matrix Waug[(in+1), pitch(out)] whose last row is the
//    bias -- the reference's own weight order (W then b) already is that matrix;
//    every activation buffer carries a constant 1.0 in column `in`, so bias add
//    (forward) and bias gradient (backward) fall out of the GEMMs themselves.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define MRGAN_TID_Z 5   // noise stream ids 0..4 = GaussianNoise layers of D, 5 = z
#define MRGAN_TID_GEN 6 // z of mrgan_generate / mrgan_sample_stats (step word = the caller's seed); no training stream uses it

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_SOFTPLUS = 2, ACT_LEAKY = 3 };   // ACT_LEAKY: LeakyReLU(alpha), others/wganlpctsemi.py:169
enum { EPI_FWD = 0, EPI_DX = 1, EPI_STORE = 2 };

// Per-fold device state.  One per fold, resident in HBM for the handle's life.
struct FoldState {
  uint32_t key0, key1;   // Philox key (from mrgan_fold_shape.seed)
  int iterations;        // Keras `adam.iterations`, shared by D and G (mr_gan.py:165-167)
  int it_net[2];         // per-net counters used when shared_t == 0
  int rng_step;          // number of executed train steps = Philox `step` word
  float lr_t[2];         // lr * sqrt(1-b2^t) / (1-b1^t) of the D step / G step in flight (per net: the D net's
                         // dW+Adam kernels may still run while the next G step's batch assembly writes its own value)
  int D, n_train, n_test;
  int ldx;               // pitch of x_train
  const float* x_train;  // [n_train, ldx] scaled features (device-resident fold data)
  const int* y_train;    // [n_train]
  const int* y_test;     // [n_test]
  const int* idx[3];     // epoch row indices: labeled, unlabeled (D step), unlabeled (G step)
  const float* stage_x;  // [3B, ldx] host-provided batches of the step API
  const int* stage_y;    // [B]
  const float* stage_z;  // [B, noise_dim]
  float* a0; int lda0;   // stacked, noisy D input [3B, pitch(D+1)]
  float* z;  int ldz;    // generator input [B, pitch(noise_dim+1)]
  int* labels_cur;       // [B] labels of the labeled rows of the step in flight
};

// One GEMM of the step, for one fold: C[M,N] = op(A)[M,K] * op(B)[K,N] (+ epilogue).
struct GemmDesc {
  const float* A; const float* B; float* C; float* C2; const float* aux;
  int lda, ldb, ldc, ldc2, ldaux;
  int M, N, K;
  int act, epi;
  float sigma; int tid; int row0;   // noise added to C2: sigma * n(row0 + m, n)
  int fold;
  int rnd;                          // tf32 mode: bit 0 / bit 1 = round C / C2 to tf32 (they feed a tcgen05 MMA)
};

// Per-step constants passed by value to the kernels: Adam hyper-parameters and, for the data-parallel mode, the
// batch geometry (dp_bloc rows per section on this rank, dp_bg rows per section globally, this rank's index).
struct AdamHyper {
  float lr, b1, b2, eps; int shared_t; int dp_bloc, dp_bg, dp_rank;
  // constants of the loss / BatchNorm heads fused into GEMM epilogues, and the batch index of the step being enqueued
  float w_unl, bn_eps; int n_classes, t;
  // discriminator variants of others/wganlpctsemi.py:166-179: LeakyReLU slope, and Dropout(rate) in place of the
  // GaussianNoise layers between hidden layers (drop == 0: the reference's GaussianNoise); drop_inv = 1 / (1 - drop)
  float alpha, drop, drop_inv;
};

// Stacked-row index of this rank -> stacked-row index of the GLOBAL batch (identity unless data-parallel): sections
// [labeled | unlabeled | fake] of dp_bg rows each, of which this rank holds rows [rank*bloc, (rank+1)*bloc).  The noise
// stream is keyed by the global index, so W ranks draw exactly what one GPU would draw for the same global batch.
// dp_rank < 0 selects the VIRTUAL-rank mode (mrgan_dp_init_virtual): the folds of one handle play the ranks, so the rank
// of a row is the index of the fold it belongs to -- the whole data-parallel path then runs, and is tested, on ONE GPU.
__host__ __device__ inline int global_row(int L, const AdamHyper& hp, int fold = 0) {
  if (hp.dp_bg == hp.dp_bloc) return L;
  const int sec = L / hp.dp_bloc;
  return sec * hp.dp_bg + (hp.dp_rank < 0 ? fold : hp.dp_rank) * hp.dp_bloc + (L - sec * hp.dp_bloc);
}

// row pitch in elements: a multiple of 8 so that both the fp32 rows and their fp16 operand copies have 16-byte strides (TMA)
__host__ __device__ inline int pitch8(int w) { return (w + 7) & ~7; }

// ---------------------------------------------------------------- Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Box-Muller on the four words of one Philox output: the 4 normals of rows 4*rowgroup .. 4*rowgroup+3
__device__ __forceinline__ void box_muller4(const uint4 x, float out[4]) {
  const float s = 1.1920928955078125e-07f;   // 2^-23
  const float u1a = ((float)(x.x >> 9) + 0.5f) * s, u2a = ((float)(x.y >> 9) + 0.5f) * s;
  const float u1b = ((float)(x.z >> 9) + 0.5f) * s, u2b = ((float)(x.w >> 9) + 0.5f) * s;
  // fast-math intrinsics: |error| of a normal <= ~3e-6 (lg2.approx / sin.approx / cos.approx on [-pi, pi], sqrt.approx), far
  // below the 1e-3 loss tolerance; the epilogue warps generate ~800k normals per fold and step pair
  // ln u = lg2.approx(u) * ln 2: what __logf computes, minus its subnormal-input handling (u >= 2^-24 here) -- same bits
  const float ra = sqrt_approx(-2.0f * (lg2_approx(u1a) * 0.693147182464599609375f)), rb = sqrt_approx(-2.0f * (lg2_approx(u1b) * 0.693147182464599609375f));
  const float pi = 3.14159265358979323846f;
  const float ta = pi * (2.0f * u2a - 1.0f), tb = pi * (2.0f * u2b - 1.0f);
  const float sa = __sinf(ta), ca = __cosf(ta), sb = __sinf(tb), cb = __cosf(tb);
  out[0] = ra * ca; out[1] = ra * sa; out[2] = rb * cb; out[3] = rb * sb;
}

// The 4 normals of rows 4*rowgroup .. 4*rowgroup+3 at column `col`
// (definition: oracle/philox.py module docstring).
__device__ __forceinline__ void normal4(uint32_t k0, uint32_t k1, uint32_t rowgroup, uint32_t col,
                                        uint32_t step, uint32_t tid, float out[4]) {
  box_muller4(philox4x32_10(make_uint4(rowgroup, col, step, tid), k0, k1), out);
}

// Dropout(rate) keep factors of the same four rows from the same four words: u_i = ((x_i >> 9) + 0.5) 2^-23, kept (factor
// 1 / (1 - rate)) iff u_i >= rate (definition: oracle/philox.py:dropout_factor).
__device__ __forceinline__ void keep4(const uint4 x, float rate, float inv, float out[4]) {
  const float s = 1.1920928955078125e-07f;   // 2^-23
  out[0] = (((float)(x.x >> 9) + 0.5f) * s >= rate) ? inv : 0.f;
  out[1] = (((float)(x.y >> 9) + 0.5f) * s >= rate) ? inv : 0.f;
  out[2] = (((float)(x.z >> 9) + 0.5f) * s >= rate) ? inv : 0.f;
  out[3] = (((float)(x.w >> 9) + 0.5f) * s >= rate) ? inv : 0.f;
}
// what a forward epilogue combines with the activation of rows 4*rowgroup..+3: N(0,1) draws (y = x + sigma n) or, with
// drop > 0, dropout keep factors (y = x f).  ONE Philox evaluation either way (the counter stream is shared).
__device__ __forceinline__ void noise_or_drop4(uint32_t k0, uint32_t k1, uint32_t rowgroup, uint32_t col, uint32_t step, uint32_t tid,
                                               float drop, float inv, float out[4]) {
  const uint4 x = philox4x32_10(make_uint4(rowgroup, col, step, tid), k0, k1);
  if (drop > 0.f) keep4(x, drop, inv, out);
  else box_muller4(x, out);
}

// Out-of-line noise draws for the GEMM epilogues: they draw up to 38 row groups per thread from several places, and an
// inlined Philox (~150 instructions, plus the integer division of global_row) per call site grew the forward kernel to
// 9 k instructions = 146 KB of SASS, far beyond the instruction cache -- the epilogue loop was fetching its own code
// from L2 (ncu: no_inst stalls).  One call per row group; with 2 epilogue warps per scheduler a single Philox chain per
// warp already keeps the issue slots busy.  `local_row` is this rank's stacked row index (see global_row).
__device__ __noinline__ float4 noise4_call(uint32_t k0, uint32_t k1, int local_row, uint32_t col, uint32_t step, uint32_t tid,
                                           int dp_bloc, int dp_bg, int dp_rank, float drop, float inv) {
  AdamHyper hp; hp.dp_bloc = dp_bloc; hp.dp_bg = dp_bg; hp.dp_rank = dp_rank;
  float n[4];
  noise_or_drop4(k0, k1, (uint32_t)global_row(local_row, hp) >> 2, col, step, tid, drop, inv, n);
  return make_float4(n[0], n[1], n[2], n[3]);
}
// one element (a 4-row group that straddles a section / rank boundary is drawn element by element)
__device__ __noinline__ float noise1_call(uint32_t k0, uint32_t k1, int local_row, uint32_t col, uint32_t step, uint32_t tid,
                                          int dp_bloc, int dp_bg, int dp_rank, float drop, float inv) {
  AdamHyper hp; hp.dp_bloc = dp_bloc; hp.dp_bg = dp_bg; hp.dp_rank = dp_rank;
  const uint32_t gr = (uint32_t)global_row(local_row, hp);
  float n[4];
  noise_or_drop4(k0, k1, gr >> 2, col, step, tid, drop, inv, n);
  const uint32_t e = gr & 3u;
  return e == 0 ? n[0] : (e == 1 ? n[1] : (e == 2 ? n[2] : n[3]));
}

__device__ __forceinline__ float normal1(uint32_t k0, uint32_t k1, uint32_t row, uint32_t col,
                                         uint32_t step, uint32_t tid) {
  float n[4];
  normal4(k0, k1, row >> 2, col, step, tid, n);
  return n[row & 3];
}

// Round-to-nearest onto the tf32 grid (10 mantissa bits).  kind::tf32 MMAs TRUNCATE their fp32 operands;
// an operand that already sits on the grid passes through unchanged, so producers round (unbiased) once.
__device__ __forceinline__ float rna_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// How a kernel stores a value that the next tensor-core GEMM reads as an operand (precision mode of the handle):
//   mode 0 (fp32 path)  : as is
//   mode 1 (tf32)       : rounded to nearest onto the tf32 grid, in place
//   mode 2 (f16)        : rounded to nearest to fp16 into the SHADOW arena -- one __half per float of the handle's arena
//                         at the same element index (hbase[p - fbase]), so pitches and descriptor offsets carry over.
//                         Gradient-side operands (dZ) are stored multiplied by the loss scale `gscale` (a power of two;
//                         every consumer is linear, the Adam update divides it out again) and saturate at the largest
//                         fp16 instead of overflowing to infinity.  (kind::f16 does not take an f16 operand together with
//                         a bf16 one -- measured: illegal instruction -- so unscaled bf16 gradients are not an option
//                         while weights and activations are fp16.)
struct OperandMode { int mode; float gscale; const float* fbase; __half* hbase; };

#define MRGAN_F16_LOSS_SCALE 4096.0f

__device__ __forceinline__ __half grad_to_half(float x) { return __float2half_rn(fminf(fmaxf(x, -65504.0f), 65504.0f)); }

__device__ __forceinline__ void put_operand(float* p, float x, const OperandMode& om) {
  if (om.mode == 2) om.hbase[p - om.fbase] = __float2half_rn(x);
  else *p = (om.mode == 1) ? rna_tf32(x) : x;
}
// gradient-side operand produced from an UNSCALED value (loss heads, BatchNorm backward)
__device__ __forceinline__ void put_grad_operand(float* p, float x, const OperandMode& om) {
  if (om.mode == 2) om.hbase[p - om.fbase] = grad_to_half(x * om.gscale);
  else put_operand(p, x, om);
}

// kind::tf32 truncates the fp32 master weights it reads: w -> w (1 - e), e in [0, 2^-10).  For mantissas
// that are log-uniform (any smooth distribution over a few octaves) E[e] = 2^-11 / (2 ln 2) = 3.52e-4, for
// uniform mantissas 2^-11 ln 2 = 3.38e-4.  Every pre-activation therefore shrinks by ~3.45e-4 per layer (a
// systematic 2e-3 on the 6-layer logits and on the feature-matching loss).  The forward / dX epilogues of the
// tf32 path multiply the accumulator by this constant, which removes the mean and leaves a zero-mean error of
// ~2e-4 per pre-activation.  Activation / gradient operands are rounded to nearest by their producers instead.
#define TF32_TRUNC_DEBIAS 1.000345f

__device__ __forceinline__ float softplusf(float x) {
  // log(1+e^x), stable on both tails (K.softplus)
  return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x)));
}

// tensor-core path: two MUFU ops instead of the libm expf / log1pf sequences (which unroll to ~100 instructions per
// element in the GEMM epilogues); |error| < 1e-7 absolute: log(1 + e) by its series where 1 + e would round
__device__ __forceinline__ float softplus_fast(float x) {
  const float e = __expf(-fabsf(x));
  const float l = e < 1e-3f ? e * fmaf(e, fmaf(e, 0.33333333f, -0.5f), 1.0f) : __logf(1.0f + e);
  return fmaxf(x, 0.0f) + l;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum, result valid in thread 0; `sh` needs 32 floats
__device__ __forceinline__ float block_sum(float v, float* sh) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    v = (l < (int)((blockDim.x + 31) >> 5)) ? sh[l] : 0.0f;
    v = warp_sum(v);
  }
  return v;
}
