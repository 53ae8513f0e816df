// kernels_simt.cuh -- fp32 (FFMA) kernels of the training step: grouped GEMM with fused
// epilogues, batch assembly + noise, BatchNorm, loss heads, feature matching, flat Adam.
// All kernels are grouped over folds through blockIdx.z (or .y) and read their
// per-fold operands from descriptor tables that live in HBM for the handle's life.
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------ grouped GEMM (fp32)
// C[M,N] = op(A)[M,K] * op(B)[K,N]; 64x64x16 tiles, 256 threads, 4x4 micro-tiles,
// register-prefetch double buffering.
//   AT = false: A stored [M, lda] (K contiguous)   AT = true: A stored [K, lda] (M contiguous)
//   BT = false: B stored [K, ldb] (N contiguous)   BT = true: B stored [N, ldb] (K contiguous)
// forward  (mr_gan.py:111-128 Dense):   NN  act(A @ Waug)            (+ GaussianNoise for the next layer)
// backward dX:                          NT  (dZ @ Waug[:in]^T) * act'(h)
// backward dW,db:                       TN  A_aug^T @ dZ            (last row = bias gradient)
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

template <bool AT, bool BT>
__global__ void __launch_bounds__(256)
k_gemm_simt(const GemmDesc* __restrict__ descs, const FoldState* __restrict__ folds, int rows_override, AdamHyper hp) {
  const GemmDesc d = descs[blockIdx.z];
  int M = d.M, K = d.K;
  const int N = d.N;
  if (rows_override > 0) { if (AT) K = rows_override; else M = rows_override; }
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  if (m0 >= M || n0 >= N) return;

  __shared__ __align__(16) float As[2][16][68];
  __shared__ __align__(16) float Bs[2][16][68];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

  auto load_a = [&](int k0) -> float4 {
    if (AT) {
      const int k = k0 + (tid >> 4), m = m0 + (tid & 15) * 4;
      return (k < K && m < d.lda) ? ldg4(d.A + (size_t)k * d.lda + m) : zero4;
    } else {
      const int m = m0 + (tid >> 2), k = k0 + (tid & 3) * 4;
      return (m < M && k < d.lda) ? ldg4(d.A + (size_t)m * d.lda + k) : zero4;
    }
  };
  auto load_b = [&](int k0) -> float4 {
    if (!BT) {
      const int k = k0 + (tid >> 4), n = n0 + (tid & 15) * 4;
      return (k < K && n < d.ldb) ? ldg4(d.B + (size_t)k * d.ldb + n) : zero4;
    } else {
      const int n = n0 + (tid >> 2), k = k0 + (tid & 3) * 4;
      return (n < N && k < d.ldb) ? ldg4(d.B + (size_t)n * d.ldb + k) : zero4;
    }
  };
  auto store_a = [&](int buf, float4 v) {
    if (AT) {
      *reinterpret_cast<float4*>(&As[buf][tid >> 4][(tid & 15) * 4]) = v;
    } else {
      const int kk = (tid & 3) * 4, mm = tid >> 2;
      As[buf][kk + 0][mm] = v.x; As[buf][kk + 1][mm] = v.y; As[buf][kk + 2][mm] = v.z; As[buf][kk + 3][mm] = v.w;
    }
  };
  auto store_b = [&](int buf, float4 v) {
    if (!BT) {
      *reinterpret_cast<float4*>(&Bs[buf][tid >> 4][(tid & 15) * 4]) = v;
    } else {
      const int kk = (tid & 3) * 4, nn = tid >> 2;
      Bs[buf][kk + 0][nn] = v.x; Bs[buf][kk + 1][nn] = v.y; Bs[buf][kk + 2][nn] = v.z; Bs[buf][kk + 3][nn] = v.w;
    }
  };

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int nk = (K + 15) >> 4;
  float4 ra = load_a(0), rb = load_b(0);
  store_a(0, ra); store_b(0, rb);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int buf = kt & 1;
    const bool more = (kt + 1 < nk);
    if (more) { ra = load_a((kt + 1) << 4); rb = load_b((kt + 1) << 4); }
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (more) { store_a(buf ^ 1, ra); store_b(buf ^ 1, rb); }
    __syncthreads();
  }

  // ---- epilogue ----
  const int mb = m0 + ty * 4, nb = n0 + tx * 4;
  if (d.epi == EPI_STORE) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = mb + i;
      if (m >= M) break;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (nb + j < N) d.C[(size_t)m * d.ldc + nb + j] = acc[i][j];
    }
    return;
  }
  if (d.epi == EPI_DX) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = mb + i;
      if (m >= M) break;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = nb + j;
        if (n >= N) continue;
        float v = acc[i][j];
        if (d.act == ACT_RELU || d.act == ACT_LEAKY) {       // aux = h, or with a Dropout layer behind the activation its dropped output
          const float a = d.aux[(size_t)m * d.ldaux + n];
          const bool drop = hp.drop > 0.f && d.tid >= 1;
          float mlt = (a > 0.f ? 1.0f : (d.act == ACT_LEAKY ? hp.alpha : 0.f)) * (drop ? hp.drop_inv : 1.0f);
          if (drop && a == 0.f) mlt = 0.f;
          v *= mlt;
        } else if (d.act == ACT_SOFTPLUS) v *= 1.0f - expf(-d.aux[(size_t)m * d.ldaux + n]);
        d.C[(size_t)m * d.ldc + n] = v;
      }
    }
    return;
  }
  // EPI_FWD: activation, optional clean copy (C), optional noisy copy for the next layer (C2)
  const bool mul = hp.drop > 0.f && d.C2 != nullptr && d.tid >= 1;      // Dropout in place of GaussianNoise (hidden layers)
  const float ddrop = mul ? hp.drop : 0.f;
  const bool noisy = (d.C2 != nullptr) && (d.sigma != 0.f || mul);
  uint32_t k0 = 0, k1 = 0, step = 0;
  if (noisy) { const FoldState& fs = folds[d.fold]; k0 = fs.key0; k1 = fs.key1; step = (uint32_t)fs.rng_step; }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = nb + j;
    if (n >= N) continue;
    float nz[4] = {0.f, 0.f, 0.f, 0.f};
    if (noisy) {
      if (((d.row0 + mb) & 3) == 0 && (hp.dp_bg == hp.dp_bloc || (hp.dp_bloc & 3) == 0)) {
        noise_or_drop4(k0, k1, (uint32_t)global_row(d.row0 + mb, hp, d.fold) >> 2, (uint32_t)n, step, (uint32_t)d.tid, ddrop, hp.drop_inv, nz);
      } else {
        for (int i = 0; i < 4; ++i) {
          const uint32_t gr = (uint32_t)global_row(d.row0 + mb + i, hp, d.fold);
          float q[4];
          noise_or_drop4(k0, k1, gr >> 2, (uint32_t)n, step, (uint32_t)d.tid, ddrop, hp.drop_inv, q);
          nz[i] = q[gr & 3];
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = mb + i;
      if (m >= M) continue;
      float v = acc[i][j];
      if (d.act == ACT_RELU) v = fmaxf(v, 0.f);
      else if (d.act == ACT_SOFTPLUS) v = softplusf(v);
      else if (d.act == ACT_LEAKY) v = v > 0.f ? v : hp.alpha * v;
      if (d.C) d.C[(size_t)m * d.ldc + n] = v;
      if (d.C2) d.C2[(size_t)m * d.ldc2 + n] = mul ? v * nz[i] : v + d.sigma * nz[i];
    }
  }
}

// ------------------------------------------------------------------ batch assembly
// Builds the stacked, noisy discriminator input and the generator input of one step
// (replaces the numpy slicing + np.random.normal of mr_gan.py:206-207,212-213 and the
// first GaussianNoise layer mr_gan.py:118) and computes Adam's lr_t for the step.
//   mode 0 (D step): rows [0,B) labeled, [B,2B) unlabeled; rows [2B,3B) come from G
//   mode 1 (G step): rows [B,2B) unlabeled; rows [0,B) come from G
//   mode 2 (mr_nn step): rows [0,n) labeled
// from_stage: rows come from the step-API staging buffers instead of the resident fold.
// PG: 4-row noise groups per thread: 2 at the reference batch (a fold's batch is ~100 rows, and 13 x 10 blocks per fold keep
// the grid large enough), 4 in the large-batch regime.
template <int PG>
__global__ void __launch_bounds__(128)
k_prep(FoldState* __restrict__ folds, int fold_base, int mode, int from_stage, int t, int B, int nrows,
       int noise_dim, float sigma_in, AdamHyper hp, OperandMode om) {
  FoldState& fs = folds[fold_base + blockIdx.z];
  const int c = blockIdx.x * 128 + threadIdx.x;
  const uint32_t step = (uint32_t)fs.rng_step;
  const int D = fs.D;

  if (blockIdx.x == 0 && blockIdx.y == 0) {
    if (threadIdx.x == 0) {
      const int net = (mode == 1) ? 1 : 0;
      const int tt = (hp.shared_t ? fs.iterations : fs.it_net[net]) + 1;
      const double b1t = pow((double)hp.b1, (double)tt), b2t = pow((double)hp.b2, (double)tt);
      fs.lr_t[net] = (float)((double)hp.lr * sqrt(1.0 - b2t) / (1.0 - b1t));
    }
    if (mode != 1) {
      for (int r = threadIdx.x; r < (mode == 2 ? nrows : B); r += 128)
        fs.labels_cur[r] = from_stage ? fs.stage_y[r] : fs.y_train[fs.idx[0][(size_t)t * B + r]];
    }
  }

  const bool aligned = (hp.dp_bloc & 3) == 0 || hp.dp_bg == hp.dp_bloc;   // 4-row noise groups stay inside one section
  const int fold = fold_base + (int)blockIdx.z;
  // rows that this step assembles from the data set: mode 0 -> [0, 2B), mode 1 -> [B, 2B), mode 2 -> [0, nrows)
  const int r_lo = (mode == 1) ? B : 0, r_hi = (mode == 2) ? nrows : min(nrows, 2 * B);
  // A thread assembles PG row groups of 4 rows of one column: the gathers of all of them are issued first, then their
  // Philox chains run interleaved in pairs (one chain per thread left this kernel latency-bound)
  const int rg = blockIdx.y;
  const int blk_lo = rg * PG * 4;
  // Interior block (all but one or two blocks per fold and section): every row of the block is assembled, from ONE section,
  // in whole noise groups -- no clamps, no per-row predicates, one index stream, operand format hoisted out of the row loop.
  // With the generic path below the kernel issued ~78 instructions per element against ~27 of Philox + Box-Muller.
  const bool interior = aligned && blk_lo >= r_lo && blk_lo + PG * 4 <= r_hi &&
                        (mode == 2 || blk_lo / B == (blk_lo + PG * 4 - 1) / B);
  if (c < D && interior) {
    const int sec = (mode != 2 && blk_lo >= B) ? 1 : 0;
    const int* const idxp = fs.idx[(mode == 1) ? 2 : sec] + (size_t)t * B + (blk_lo - sec * B);
    const float* const xsrc = (from_stage ? fs.stage_x : fs.x_train) + c;
    const int ldx = fs.ldx, lda0 = fs.lda0;
    const uint32_t key0 = fs.key0, key1 = fs.key1;
    int rix[PG * 4];
    float xv[PG * 4];
    if (from_stage) {
#pragma unroll
      for (int k = 0; k < PG * 4; ++k) rix[k] = blk_lo + k;
    } else {
#pragma unroll
      for (int k = 0; k < PG * 4; ++k) rix[k] = __ldg(idxp + k);
    }
#pragma unroll
    for (int k = 0; k < PG * 4; ++k) xv[k] = __ldg(xsrc + (size_t)rix[k] * ldx);
    float* const dst = fs.a0 + (size_t)blk_lo * lda0 + c;
    __half* const hdst = om.mode == 2 ? om.hbase + (dst - om.fbase) : nullptr;
#pragma unroll
    for (int u0 = 0; u0 < PG; u0 += 2) {
      float nz[2][4];
#pragma unroll
      for (int v = 0; v < 2; ++v)
        normal4(key0, key1, (uint32_t)global_row(blk_lo + 4 * (u0 + v), hp, fold) >> 2, (uint32_t)c, step, 0u, nz[v]);
#pragma unroll
      for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int k = 4 * (u0 + v) + i;
          const float y = xv[k] + sigma_in * nz[v][i];
          if (om.mode == 2) hdst[(size_t)k * lda0] = __float2half_rn(y);
          else dst[(size_t)k * lda0] = (om.mode == 1) ? rna_tf32(y) : y;
        }
    }
  } else if (c < D) {
    // generic path: edge blocks (section / batch boundaries), unaligned data-parallel row groups
    const float* const x_train = fs.x_train; const float* const stage_x = fs.stage_x;
    const int* const idx0 = fs.idx[0]; const int* const idx1 = fs.idx[1]; const int* const idx2 = fs.idx[2];
    float* const a0 = fs.a0;
    const int ldx = fs.ldx, lda0 = fs.lda0;
    const uint32_t key0 = fs.key0, key1 = fs.key1;
    float xv[PG][4];
    bool live[PG];
    // Gathers: row numbers first, then the rows, for ALL rows of the thread at once and without a branch in front of any
    // load (out-of-range rows are clamped onto a row this step does assemble and discarded at the store).  Behind per-row
    // predicates the compiler issued "index load -> wait -> row load" pairs one after the other, so a thread paid the memory
    // latency 8 times in a row: 51 % of this kernel's stall samples (profiles/r02_prep_ncu_before.txt).
    const bool blk_live = blk_lo + PG * 4 > r_lo && blk_lo < r_hi;      // uniform per block
    if (blk_live) {
      int rix[PG][4];
      if (from_stage) {
#pragma unroll
        for (int u = 0; u < PG; ++u)
#pragma unroll
          for (int i = 0; i < 4; ++i) rix[u][i] = min(max(blk_lo + 4 * u + i, r_lo), r_hi - 1);
      } else {
        const size_t tb = (size_t)t * B;
#pragma unroll
        for (int u = 0; u < PG; ++u)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = min(max(blk_lo + 4 * u + i, r_lo), r_hi - 1);
            const int* const idx = (mode == 1) ? idx2 : ((mode == 0 && r >= B) ? idx1 : idx0);
            const int lr = (mode == 2) ? r : (r < B ? r : r - B);
            rix[u][i] = __ldg(idx + tb + lr);
          }
      }
      const float* const xsrc = (from_stage ? stage_x : x_train) + c;
#pragma unroll
      for (int u = 0; u < PG; ++u)
#pragma unroll
        for (int i = 0; i < 4; ++i) xv[u][i] = __ldg(xsrc + (size_t)rix[u][i] * ldx);
    }
#pragma unroll
    for (int u = 0; u < PG; ++u) {
      const int g4 = blk_lo + 4 * u;
      live[u] = blk_live && g4 + 3 >= r_lo && g4 < r_hi;
    }
#pragma unroll
    for (int u0 = 0; u0 < PG; u0 += 2) {
      float nz[2][4];
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int g4 = (rg * PG + u0 + v) * 4;
        if (!live[u0 + v]) continue;
        if (aligned) normal4(key0, key1, (uint32_t)global_row(g4, hp, fold) >> 2, (uint32_t)c, step, 0u, nz[v]);
        else for (int i = 0; i < 4; ++i) nz[v][i] = normal1(key0, key1, (uint32_t)global_row(g4 + i, hp, fold), (uint32_t)c, step, 0u);
      }
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int g4 = (rg * PG + u0 + v) * 4;
        if (!live[u0 + v]) continue;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = g4 + i;
          if (r < r_lo || r >= r_hi) continue;
          put_operand(a0 + (size_t)r * lda0 + c, xv[u0 + v][i] + sigma_in * nz[v][i], om);
        }
      }
    }
  }
  if (mode != 2 && c < noise_dim) {       // generator input z (mr_gan.py:206,212)
    for (int u = 0; u < PG; ++u) {
      const int g4 = (rg * PG + u) * 4;
      if (g4 >= B) break;
      float nz[4] = {0.f, 0.f, 0.f, 0.f};
      if (!from_stage) {
        if (aligned) normal4(fs.key0, fs.key1, (uint32_t)global_row(g4, hp, fold) >> 2, (uint32_t)c, step, MRGAN_TID_Z, nz);
        else for (int i = 0; i < 4; ++i) nz[i] = normal1(fs.key0, fs.key1, (uint32_t)global_row(g4 + i, hp, fold), (uint32_t)c, step, MRGAN_TID_Z);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = g4 + i;
        if (r >= B) break;
        const float v = from_stage ? fs.stage_z[(size_t)r * noise_dim + c] : nz[i];
        put_operand(fs.z + (size_t)r * fs.ldz + c, v, om);
      }
    }
  }
}

// ------------------------------------------------------------------ BatchNorm (batch statistics)
struct BnDesc {
  const float* h1; float* xhat; float* u; float* istd;      // fwd
  const float* gamma; const float* beta;
  const float* du; float* dz1; float* g_gamma; float* g_beta;  // bwd
  int ld, ldu, B, W;
};

// mr_gan.py:112 BatchNormalization(epsilon=2e-5) in training phase: biased batch variance.
// Block = 32 columns x 8 row slices (256 threads): the batch loop is split 8 ways and reduced through shared memory,
// so the dependent-load chain per thread is B/8 rows instead of B.
// The slice count is blockDim.x / 32: 8 at the reference batch, 32 in the large-batch regime.
#define BN_COLS 32
#define BN_MAX_SLICES 32
__global__ void __launch_bounds__(1024) k_bn_fwd(const BnDesc* __restrict__ descs, float eps, OperandMode om) {
  __shared__ float red[2][BN_MAX_SLICES][BN_COLS];
  const BnDesc d = descs[blockIdx.z];
  const int BN_SLICES = blockDim.x / BN_COLS;
  const int cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  const bool ok = j < d.W;
  float s = 0.f;
  if (ok) for (int r = sl; r < d.B; r += BN_SLICES) s += d.h1[(size_t)r * d.ld + j];
  red[0][sl][cx] = s;
  __syncthreads();
  float mu = 0.f;
  for (int i = 0; i < BN_SLICES; ++i) mu += red[0][i][cx];
  mu /= d.B;
  float q = 0.f;
  if (ok) for (int r = sl; r < d.B; r += BN_SLICES) { const float x = d.h1[(size_t)r * d.ld + j] - mu; q = fmaf(x, x, q); }
  red[1][sl][cx] = q;
  __syncthreads();
  float var = 0.f;
  for (int i = 0; i < BN_SLICES; ++i) var += red[1][i][cx];
  if (!ok) return;
  const float istd = rsqrtf(var / d.B + eps);
  if (sl == 0) d.istd[j] = istd;
  const float g = d.gamma[j], b = d.beta[j];
  for (int r = sl; r < d.B; r += BN_SLICES) {
    const float xh = (d.h1[(size_t)r * d.ld + j] - mu) * istd;
    d.xhat[(size_t)r * d.ld + j] = xh;
    const float u = fmaf(g, xh, b);
    put_operand(d.u + (size_t)r * d.ldu + j, u, om);
  }
}

// BN backward + softplus' of the layer in front of it (G layer 1): du -> dgamma, dbeta, dz1.
__global__ void __launch_bounds__(1024) k_bn_bwd(const BnDesc* __restrict__ descs, OperandMode om) {
  __shared__ float red[2][BN_MAX_SLICES][BN_COLS];
  const BnDesc d = descs[blockIdx.z];
  const int BN_SLICES = blockDim.x / BN_COLS;
  const int cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  const bool ok = j < d.W;
  const float ginv = (om.mode == 2) ? 1.0f / om.gscale : 1.0f;      // f16 mode: du arrives multiplied by the loss scale
  float p1 = 0.f, p2 = 0.f;
  if (ok) for (int r = sl; r < d.B; r += BN_SLICES) {
    const float du = d.du[(size_t)r * d.ld + j] * ginv;
    p1 += du;
    p2 = fmaf(du, d.xhat[(size_t)r * d.ld + j], p2);
  }
  red[0][sl][cx] = p1; red[1][sl][cx] = p2;
  __syncthreads();
  float s1 = 0.f, s2 = 0.f;
  for (int i = 0; i < BN_SLICES; ++i) { s1 += red[0][i][cx]; s2 += red[1][i][cx]; }
  if (!ok) return;
  if (sl == 0) {      // f16 mode: the whole gradient buffer carries the loss scale (k_adam divides it out)
    const float gs = (om.mode == 2) ? om.gscale : 1.0f;
    d.g_gamma[j] = s2 * gs; d.g_beta[j] = s1 * gs;
  }
  const float g = d.gamma[j], istd = d.istd[j], invB = 1.0f / d.B;
  for (int r = sl; r < d.B; r += BN_SLICES) {
    const float xh = d.xhat[(size_t)r * d.ld + j];
    const float dxh = d.du[(size_t)r * d.ld + j] * ginv * g;
    const float dh1 = istd * (dxh - invB * g * s1 - xh * invB * g * s2);
    const float dz = dh1 * (1.0f - expf(-d.h1[(size_t)r * d.ld + j]));
    put_grad_operand(d.dz1 + (size_t)r * d.ld + j, dz, om);
  }
}

// ------------------------------------------------------------------ loss heads
#define LOSS_MAX_BLOCKS 64
struct LossDesc {
  const float* logits; float* dlogits; int ld;   // [rows, ld]
  const int* labels;
  const float* mid; float* dmid; int ldmid, lddmid, Wmid;   // feature matching
};

// Salimans-style supervised + unsupervised losses on the stacked logits
// (mr_gan.py:146-149,161) and their gradients (SURVEY.md 3.2).
// gridDim.x == 1 at the reference batch.  In the large-batch regime the 3B rows are spread over gridDim.x blocks (one block
// walked 24 576 rows in 184 us); each block leaves its three partial sums in `part` ([fold][block][4]) and the last one to
// arrive (`ctr[fold]`) adds them in block order, so the statistics stay reproducible.
__global__ void __launch_bounds__(256)
k_loss_disc(const LossDesc* __restrict__ descs, float* __restrict__ step_stats, int fold_base, int nf_total,
            int t, int B, int K, float w_unl, OperandMode om, int Bg, float* __restrict__ part, unsigned* __restrict__ ctr) {
  __shared__ float sh[32];
  const LossDesc d = descs[blockIdx.z];   // B rows per section on this rank, Bg in the global batch (means are over Bg)
  float s_lab = 0.f, s_unl = 0.f, s_err = 0.f;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < 3 * B; r += blockDim.x * gridDim.x) {
    const float* l = d.logits + (size_t)r * d.ld;
    float mx = l[0]; int am = 0;
    for (int k = 1; k < K; ++k) if (l[k] > mx) { mx = l[k]; am = k; }
    float se = 0.f;
    for (int k = 0; k < K; ++k) se += expf(l[k] - mx);
    const float lse = mx + logf(se), inv = 1.0f / se;
    float* dl = d.dlogits + (size_t)r * d.ld;
    if (r < B) {
      const int y = d.labels[r];
      s_lab += lse - l[y];
      s_err += (am != y) ? 1.f : 0.f;
      for (int k = 0; k < K; ++k) {
        const float g = (expf(l[k] - mx) * inv - (k == y ? 1.f : 0.f)) / Bg;
        put_grad_operand(dl + k, g, om);
      }
    } else {
      const float sp = softplusf(lse), sg = 1.0f / (1.0f + expf(-lse));
      float coef;
      if (r < 2 * B) { s_unl += 0.5f * (sp - lse); coef = 0.5f * (sg - 1.0f); }
      else           { s_unl += 0.5f * sp;         coef = 0.5f * sg; }
      coef *= w_unl / Bg;
      for (int k = 0; k < K; ++k) {
        const float g = coef * expf(l[k] - mx) * inv;
        put_grad_operand(dl + k, g, om);
      }
    }
  }
  s_lab = block_sum(s_lab, sh);
  s_unl = block_sum(s_unl, sh);
  s_err = block_sum(s_err, sh);
  float* const st = step_stats + ((size_t)t * nf_total + fold_base + blockIdx.z) * 4;
  if (gridDim.x == 1) {
    if (threadIdx.x == 0) { st[0] = s_lab / Bg; st[1] = s_unl / Bg; st[2] = s_err / Bg; }
    return;
  }
  float* const pf = part + (size_t)(fold_base + blockIdx.z) * 4 * LOSS_MAX_BLOCKS;
  if (threadIdx.x == 0) {
    pf[4 * blockIdx.x] = s_lab; pf[4 * blockIdx.x + 1] = s_unl; pf[4 * blockIdx.x + 2] = s_err;
    __threadfence();
    const unsigned n = atomicAdd(ctr + fold_base + blockIdx.z, 1u);
    if (n == gridDim.x - 1) {
      ctr[fold_base + blockIdx.z] = 0u;
      __threadfence();
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      for (unsigned b = 0; b < gridDim.x; ++b) { a0 += __ldcg(pf + 4 * b); a1 += __ldcg(pf + 4 * b + 1); a2 += __ldcg(pf + 4 * b + 2); }
      st[0] = a0 / Bg; st[1] = a1 / Bg; st[2] = a2 / Bg;
    }
  }
}

// Feature matching (mr_gan.py:152-154): rows [0,B) = fake, [B,2B) = real mid activations.
// Writes dZ5 (already multiplied by ReLU') for the fake rows.  1024 threads = 256 columns x 4 row slices.
__global__ void __launch_bounds__(1024)
k_fm(const LossDesc* __restrict__ descs, float* __restrict__ step_stats, int fold_base, int nf_total, int t, int B,
     OperandMode om, float alpha) {
  __shared__ float sh[32];
  __shared__ float red[2][4][256];
  const LossDesc d = descs[blockIdx.z];
  const int cx = threadIdx.x & 255, sl = threadIdx.x >> 8;
  float s = 0.f;
  for (int j0 = 0; j0 < d.Wmid; j0 += 256) {
    const int j = j0 + cx;
    const bool ok = j < d.Wmid;
    float mg = 0.f, mr = 0.f;
    if (ok) for (int r = sl; r < B; r += 4) { mg += d.mid[(size_t)r * d.ldmid + j]; mr += d.mid[(size_t)(r + B) * d.ldmid + j]; }
    __syncthreads();
    red[0][sl][cx] = mg; red[1][sl][cx] = mr;
    __syncthreads();
    if (!ok) continue;
    mg = red[0][0][cx] + red[0][1][cx] + red[0][2][cx] + red[0][3][cx];
    mr = red[1][0][cx] + red[1][1][cx] + red[1][2][cx] + red[1][3][cx];
    const float diff = (mg - mr) / B;
    if (sl == 0) s = fmaf(diff, diff, s);
    const float g = 2.0f * diff / ((float)d.Wmid * B);
    for (int r = sl; r < B; r += 4)
      put_grad_operand(d.dmid + (size_t)r * d.lddmid + j, (d.mid[(size_t)r * d.ldmid + j] > 0.f) ? g : alpha * g, om);
  }
  s = block_sum(s, sh);
  if (threadIdx.x == 0) step_stats[((size_t)t * nf_total + fold_base + blockIdx.z) * 4 + 3] = s / d.Wmid;
}

// mr_nn.py:114 loss='mse' vs one-hot, metrics=['accuracy'].
__global__ void __launch_bounds__(256)
k_loss_mse(const LossDesc* __restrict__ descs, float* __restrict__ step_stats, int fold_base, int nf_total,
           int t, int n, int rows_total, int K, OperandMode om) {
  __shared__ float sh[32];
  const LossDesc d = descs[blockIdx.z];
  float s_loss = 0.f, s_acc = 0.f;
  for (int r = n + threadIdx.x; r < rows_total; r += blockDim.x)     // ragged batch: no gradient from the unused rows
    for (int k = 0; k < K; ++k) put_grad_operand(d.dlogits + (size_t)r * d.ld + k, 0.f, om);
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
    const float* l = d.logits + (size_t)r * d.ld;
    float* dl = d.dlogits + (size_t)r * d.ld;
    const int y = d.labels[r];
    float mx = l[0]; int am = 0;
    for (int k = 1; k < K; ++k) if (l[k] > mx) { mx = l[k]; am = k; }
    float q = 0.f;
    for (int k = 0; k < K; ++k) {
      const float diff = l[k] - (k == y ? 1.f : 0.f);
      q = fmaf(diff, diff, q);
      const float g = 2.0f * diff / ((float)n * K);
      put_grad_operand(dl + k, g, om);
    }
    s_loss += q / K;
    s_acc += (am == y) ? 1.f : 0.f;
  }
  s_loss = block_sum(s_loss, sh);
  s_acc = block_sum(s_acc, sh);
  if (threadIdx.x == 0) {
    float* st = step_stats + ((size_t)t * nf_total + fold_base + blockIdx.z) * 4;
    st[0] = s_loss / n; st[1] = s_acc / n;
  }
}


// ------------------------------------------------------------------ data-parallel variants (statistics / apply split)
// In the data-parallel mode the batch statistics that the reference takes over the whole batch (BatchNorm mean /
// variance mr_gan.py:112, feature-matching means mr_gan.py:152-153) are summed locally, all-reduced over NVLink,
// and applied by a second kernel, so that W ranks compute exactly the single-GPU large-batch step.
// part / ctr: scratch of the row-parallel statistics kernels -- SPLIT_MAX_Y row chunks x 2 x 512 partial sums per fold, and
// one arrival counter per column block (the last block to arrive adds the chunks IN CHUNK ORDER and resets the counter,
// so the sums are reproducible and the kernels replay inside a CUDA graph).
struct DpBufs { float* bnf; float* bnb; float* fm; float* part; unsigned* ctr; };   // per fold: [2*W] sums each (W = 500 / 500 / 250)
#define SPLIT_MAX_Y 32
#define SPLIT_PART_W 512

// Publishes this block's partial sums (already written by its slice-0 threads) and tells whether it is the last of the
// gridDim.y row-chunk blocks of its column block to do so.  Block-uniform result.
__device__ __forceinline__ bool split_last_block(unsigned* ctr) {
  __shared__ int last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned n = atomicAdd(ctr, 1u);
    last = (n == gridDim.y - 1);
    if (last) *ctr = 0u;
  }
  __syncthreads();
  if (last) __threadfence();
  return last != 0;
}

// Column sums of two quantities over this block's row chunk -> out[j], out[W + j] (gridDim.y == 1) or, with several row
// chunks, the chunk's partial; the last block adds the partials in chunk order.  `red` = [2][slices][32] shared floats.
__device__ __forceinline__ void split_reduce(float a, float b, float (*red)[BN_MAX_SLICES][BN_COLS], int W, const DpBufs& bf, float* out,
                                             float* out2a, float* out2b, float scale2) {
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  red[0][sl][cx] = a; red[1][sl][cx] = b;
  __syncthreads();
  if (sl == 0 && j < W) {
    a = 0.f; b = 0.f;
    for (int i = 0; i < nsl; ++i) { a += red[0][i][cx]; b += red[1][i][cx]; }
    if (gridDim.y == 1) {
      out[j] = a; out[W + j] = b;
      if (out2a) { out2a[j] = a * scale2; out2b[j] = b * scale2; }
    } else {
      float* p = bf.part + (size_t)blockIdx.y * 2 * SPLIT_PART_W;
      p[j] = a; p[SPLIT_PART_W + j] = b;
    }
  }
  if (gridDim.y == 1) return;
  if (!split_last_block(bf.ctr + blockIdx.x)) return;
  if (sl == 0 && j < W) {
    a = 0.f; b = 0.f;
    for (unsigned y = 0; y < gridDim.y; ++y) {
      const float* p = bf.part + (size_t)y * 2 * SPLIT_PART_W;
      a += __ldcg(p + j); b += __ldcg(p + SPLIT_PART_W + j);
    }
    out[j] = a; out[W + j] = b;
    if (out2a) { out2a[j] = a * scale2; out2b[j] = b * scale2; }
  }
}

// grid = (column blocks of 32, row chunks, folds); block = 32 columns x (blockDim.x / 32) row slices.  Rows of a block:
// r = blockIdx.y * slices + slice, stepping by slices * gridDim.y.
__global__ void __launch_bounds__(1024) k_bn_stats(const BnDesc* __restrict__ descs, const DpBufs* __restrict__ bufs) {
  __shared__ float red[2][BN_MAX_SLICES][BN_COLS];
  const BnDesc d = descs[blockIdx.z];
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  float s = 0.f, q = 0.f;
  if (j < d.W) for (int r = blockIdx.y * nsl + sl; r < d.B; r += nsl * gridDim.y) { const float x = d.h1[(size_t)r * d.ld + j]; s += x; q = fmaf(x, x, q); }
  split_reduce(s, q, red, d.W, bufs[blockIdx.z], bufs[blockIdx.z].bnf, nullptr, nullptr, 0.f);
}

__global__ void __launch_bounds__(1024) k_bn_apply(const BnDesc* __restrict__ descs, const DpBufs* __restrict__ bufs,
                                                   float eps, OperandMode om, int Bg) {
  const BnDesc d = descs[blockIdx.z];
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  if (j >= d.W) return;
  const float mu = bufs[blockIdx.z].bnf[j] / Bg;
  const float var = fmaxf(bufs[blockIdx.z].bnf[d.W + j] / Bg - mu * mu, 0.f);
  const float istd = rsqrtf(var + eps);
  if (sl == 0 && blockIdx.y == 0) d.istd[j] = istd;
  const float g = d.gamma[j], b = d.beta[j];
  for (int r = blockIdx.y * nsl + sl; r < d.B; r += nsl * gridDim.y) {
    const float xh = (d.h1[(size_t)r * d.ld + j] - mu) * istd;
    d.xhat[(size_t)r * d.ld + j] = xh;
    const float u = fmaf(g, xh, b);
    put_operand(d.u + (size_t)r * d.ldu + j, u, om);
  }
}

__global__ void __launch_bounds__(1024) k_bn_bwd_stats(const BnDesc* __restrict__ descs, const DpBufs* __restrict__ bufs,
                                                       OperandMode om) {
  __shared__ float red[2][BN_MAX_SLICES][BN_COLS];
  const BnDesc d = descs[blockIdx.z];
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  const float ginv = (om.mode == 2) ? 1.0f / om.gscale : 1.0f;
  float s1 = 0.f, s2 = 0.f;
  if (j < d.W) for (int r = blockIdx.y * nsl + sl; r < d.B; r += nsl * gridDim.y) { const float du = d.du[(size_t)r * d.ld + j] * ginv; s1 += du; s2 = fmaf(du, d.xhat[(size_t)r * d.ld + j], s2); }
  // bnb = [s1 | s2]; the LOCAL partial gradients g_beta = s1, g_gamma = s2 (times the loss scale of the gradient buffer):
  // the flat gradient all-reduce completes them
  split_reduce(s1, s2, red, d.W, bufs[blockIdx.z], bufs[blockIdx.z].bnb, d.g_beta, d.g_gamma, (om.mode == 2) ? om.gscale : 1.0f);
}

__global__ void __launch_bounds__(1024) k_bn_bwd_apply(const BnDesc* __restrict__ descs, const DpBufs* __restrict__ bufs,
                                                       OperandMode om, int Bg) {
  const BnDesc d = descs[blockIdx.z];
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  if (j >= d.W) return;
  const float s1 = bufs[blockIdx.z].bnb[j], s2 = bufs[blockIdx.z].bnb[d.W + j];
  const float g = d.gamma[j], istd = d.istd[j], invB = 1.0f / Bg;
  const float ginv = (om.mode == 2) ? 1.0f / om.gscale : 1.0f;
  for (int r = blockIdx.y * nsl + sl; r < d.B; r += nsl * gridDim.y) {
    const float xh = d.xhat[(size_t)r * d.ld + j];
    const float dxh = d.du[(size_t)r * d.ld + j] * ginv * g;
    const float dh1 = istd * (dxh - invB * g * s1 - xh * invB * g * s2);
    const float dz = dh1 * (1.0f - expf(-d.h1[(size_t)r * d.ld + j]));
    put_grad_operand(d.dz1 + (size_t)r * d.ld + j, dz, om);
  }
}

__global__ void __launch_bounds__(1024) k_fm_stats(const LossDesc* __restrict__ descs, const DpBufs* __restrict__ bufs, int B) {
  __shared__ float red[2][BN_MAX_SLICES][BN_COLS];
  const LossDesc d = descs[blockIdx.z];
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  float mg = 0.f, mr = 0.f;
  if (j < d.Wmid) for (int r = blockIdx.y * nsl + sl; r < B; r += nsl * gridDim.y) { mg += d.mid[(size_t)r * d.ldmid + j]; mr += d.mid[(size_t)(r + B) * d.ldmid + j]; }
  split_reduce(mg, mr, red, d.Wmid, bufs[blockIdx.z], bufs[blockIdx.z].fm, nullptr, nullptr, 0.f);
}

__global__ void __launch_bounds__(1024)
k_fm_apply(const LossDesc* __restrict__ descs, const DpBufs* __restrict__ bufs, float* __restrict__ step_stats, int fold_base,
           int nf_total, int t, int B, OperandMode om, int Bg, int world, float alpha) {
  __shared__ float sh[32];
  const LossDesc d = descs[blockIdx.z];
  const int nsl = blockDim.x / BN_COLS, cx = threadIdx.x & (BN_COLS - 1), sl = threadIdx.x / BN_COLS;
  const int j = blockIdx.x * BN_COLS + cx;
  if (j < d.Wmid) {
    const float diff = (bufs[blockIdx.z].fm[j] - bufs[blockIdx.z].fm[d.Wmid + j]) / Bg;
    const float g = 2.0f * diff / ((float)d.Wmid * Bg);
    for (int r = blockIdx.y * nsl + sl; r < B; r += nsl * gridDim.y)
      put_grad_operand(d.dmid + (size_t)r * d.lddmid + j, (d.mid[(size_t)r * d.ldmid + j] > 0.f) ? g : alpha * g, om);
  }
  if (blockIdx.x == 0 && blockIdx.y == 0) {   // the loss itself: every rank holds the same global value; the statistics block is
    float s = 0.f;                            // summed over ranks afterwards, so 1/world of it is stored
    for (int c = threadIdx.x; c < d.Wmid; c += blockDim.x) {
      const float diff = (bufs[blockIdx.z].fm[c] - bufs[blockIdx.z].fm[d.Wmid + c]) / Bg;
      s = fmaf(diff, diff, s);
    }
    s = block_sum(s, sh);
    if (threadIdx.x == 0) step_stats[((size_t)t * nf_total + fold_base + blockIdx.z) * 4 + 3] = s / d.Wmid / world;
  }
}

// ------------------------------------------------------------------ evaluation
struct EvalDesc { const float* logits; int ld; const int* y; int n; int n_batched; float* out; int* pred; };

// The predicted class of a row of logits: the FIRST maximal entry (strict > scan; a NaN never wins).  The one argmax rule
// behind both the error of k_argmax_err and the per-row predictions.
__device__ __forceinline__ int row_argmax(const float* l, int K) {
  float mx = l[0]; int am = 0;
  for (int k = 1; k < K; ++k) if (l[k] > mx) { mx = l[k]; am = k; }
  return am;
}

// test_batch (mr_gan.py:162,171): mean(argmax != y); out[0] over the first n_batched rows
// (= mean of the per-batch errors of mr_gan.py:221-223), out[1] over all rows (mr_gan.py:230),
// out[2] = mse vs one-hot over all rows (mr_nn.py:118 evaluate()[0]).  with_pred: also store every row's class in d.pred.
__global__ void __launch_bounds__(256)
k_argmax_err(const EvalDesc* __restrict__ descs, int n_override, int K, int with_pred) {
  __shared__ float sh[32];
  const EvalDesc d = descs[blockIdx.z];
  const int n = n_override > 0 ? n_override : d.n;
  const int nb = n_override > 0 ? n_override : d.n_batched;
  float e_b = 0.f, e_all = 0.f, q = 0.f;
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
    const float* l = d.logits + (size_t)r * d.ld;
    const int y = d.y[r];
    const int am = row_argmax(l, K);
    if (with_pred) d.pred[r] = am;
    for (int k = 0; k < K; ++k) { const float diff = l[k] - (k == y ? 1.f : 0.f); q = fmaf(diff, diff, q); }
    const float e = (am != y) ? 1.f : 0.f;
    e_all += e;
    if (r < nb) e_b += e;
  }
  e_b = block_sum(e_b, sh);
  e_all = block_sum(e_all, sh);
  q = block_sum(q, sh);
  if (threadIdx.x == 0) { d.out[0] = nb > 0 ? e_b / nb : 0.f; d.out[1] = e_all / n; d.out[2] = q / ((float)n * K); }
}

// Confusion counts of every fold: out[f][y][pred] over the fold's d.n rows of (d.y, d.pred); out is zeroed beforehand.
// grid (row chunks, folds); a block counts its chunk in shared memory, then adds its non-zero cells.  Integer atomics:
// the counts are exact in any order.
#define CONF_ROWS 1024
__global__ void __launch_bounds__(256) k_confusion(const EvalDesc* __restrict__ descs, int K, int* __restrict__ out) {
  __shared__ int cnt[64 * 64];
  const EvalDesc d = descs[blockIdx.y];
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) cnt[i] = 0;
  __syncthreads();
  const int r0 = blockIdx.x * CONF_ROWS, r1 = min(d.n, r0 + CONF_ROWS);
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x) atomicAdd(&cnt[d.y[r] * K + d.pred[r]], 1);
  __syncthreads();
  int* o = out + (size_t)blockIdx.y * K * K;
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) if (cnt[i]) atomicAdd(&o[i], cnt[i]);
}

// ------------------------------------------------------------------ input gradients (mrgan_input_grad / mrgan_saliency)
// Seed of the backward pass of log softmax(l)_t: d/dl = e_t - softmax(l), written over the row's phase-0 logits (read by
// nothing after the eval) in the dX operand format of the handle, like the logit gradients of k_loss_disc.  t = d.y[r], or with
// use_pred the row's predicted class (row_argmax).  One thread per row; grid (row blocks, 1, folds).
__global__ void __launch_bounds__(256)
k_logprob_seed(const EvalDesc* __restrict__ descs, int n_override, int K, int use_pred, OperandMode om) {
  const EvalDesc d = descs[blockIdx.z];
  const int n = n_override > 0 ? n_override : d.n;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  float* const l = const_cast<float*>(d.logits) + (size_t)r * d.ld;
  const int t = use_pred ? row_argmax(l, K) : d.y[r];
  float mx = l[0];
  for (int k = 1; k < K; ++k) mx = fmaxf(mx, l[k]);
  float se = 0.f;
  for (int k = 0; k < K; ++k) se += expf(l[k] - mx);
  const float inv = 1.0f / se;
  for (int k = 0; k < K; ++k) put_grad_operand(l + k, (k == t ? 1.f : 0.f) - expf(l[k] - mx) * inv, om);   // reads l[k] first
}

// f16 mode: the fp32 input gradients of OP_EX1 (C [M][ldc], N = D columns) carry the loss scale of the dX operands; ginv divides
// it out in place (a power of two: exact).  grid (blocks, 1, folds).
__global__ void __launch_bounds__(256) k_unscale_grad(const GemmDesc* __restrict__ descs, int rows_override, float ginv) {
  const GemmDesc g = descs[blockIdx.z];
  const int M = rows_override > 0 ? rows_override : g.M;
  const size_t n = (size_t)M * g.N;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    g.C[(i / g.N) * g.ldc + i % g.N] *= ginv;
}

// Saliency profile of every fold: out[f][c][j] = (1 / N_c) sum over the fold's test rows r with y_r = c of |grad[r][j]|, grad =
// the OP_EX1 output (descs[f].C, d.n rows), N_c = the number of such rows; 0 for a class without rows and for j >= D.  One
// thread per (fold, feature) and class, summing in double in row order: no atomics, so the result is bitwise reproducible and
// independent of the grouping of the folds.  grid (feature blocks, folds).
__global__ void __launch_bounds__(128)
k_saliency(const GemmDesc* __restrict__ gx, const EvalDesc* __restrict__ ev, int K, int Dmax, float* __restrict__ out) {
  const int f = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= Dmax) return;
  const GemmDesc g = gx[f];
  const EvalDesc e = ev[f];
  float* const o = out + (size_t)f * K * Dmax + j;
  for (int c = 0; c < K; ++c) {
    double s = 0.0;
    int nc = 0;
    if (j < g.N)
      for (int r = 0; r < e.n; ++r)
        if (e.y[r] == c) { s += fabs((double)g.C[(size_t)r * g.ldc + j]); ++nc; }
    o[(size_t)c * Dmax] = nc > 0 ? (float)(s / nc) : 0.f;
  }
}

// Means over the epoch's batches (mr_gan.py:215-217) -> epoch_stats[f][0..3]; [4] = batch-wise test error.
__global__ void k_epoch_reduce(const float* __restrict__ step_stats, const EvalDesc* __restrict__ evals,
                               float* __restrict__ epoch_stats, int nf, int nb, int with_eval) {
  const int f = blockIdx.x, j = threadIdx.x;
  if (j < 4) {
    float s = 0.f;
    for (int t = 0; t < nb; ++t) s += step_stats[((size_t)t * nf + f) * 4 + j];
    epoch_stats[f * 8 + j] = s / nb;
  } else if (j == 4) {
    epoch_stats[f * 8 + 4] = with_eval ? evals[f].out[0] : -1.f;
  }
}

// ------------------------------------------------------------------ flat fused Adam
// Keras-2.0.9 Adam.get_updates over one flat parameter range per fold (SURVEY.md 3.4, a8):
// m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; p -= lr_t m / (sqrt(v) + eps).
// The last block advances the fold's step counters (K.update_add(iterations, 1)).
struct AdamRange { long long off; long long n; };   // n multiple of 4, off 16B aligned

__global__ void __launch_bounds__(256)
k_adam(float* __restrict__ P, float* __restrict__ Mo, float* __restrict__ Vo, const float* __restrict__ G,
       const AdamRange* __restrict__ ranges, FoldState* __restrict__ folds, int fold_base, int net, AdamHyper hp,
       float ginv, __half* __restrict__ Ph) {      // ginv: 1 / loss scale of the gradient buffer; Ph: fp16 operand copy of P or null
  const int f = fold_base + blockIdx.y;
  const AdamRange rg = ranges[f];
  FoldState& fs = folds[f];
  const float lr_t = fs.lr_t[net];
  const float b1 = hp.b1, b2 = hp.b2, eps = hp.eps, c1 = 1.0f - hp.b1, c2 = 1.0f - hp.b2;
  const long long n4 = rg.n >> 2;
  float4* p4 = reinterpret_cast<float4*>(P + rg.off);
  float4* m4 = reinterpret_cast<float4*>(Mo + rg.off);
  float4* v4 = reinterpret_cast<float4*>(Vo + rg.off);
  const float4* g4 = reinterpret_cast<const float4*>(G + rg.off);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 p = p4[i], m = m4[i], v = v4[i];
    float4 g = __ldg(g4 + i);
    g.x *= ginv; g.y *= ginv; g.z *= ginv; g.w *= ginv;
#define ADAM1(c) m.c = fmaf(b1, m.c, c1 * g.c); v.c = fmaf(b2, v.c, c2 * g.c * g.c); p.c -= lr_t * m.c / (sqrtf(v.c) + eps);
    ADAM1(x) ADAM1(y) ADAM1(z) ADAM1(w)
#undef ADAM1
    p4[i] = p; m4[i] = m; v4[i] = v;
    if (Ph) {
      __half2* h2 = reinterpret_cast<__half2*>(Ph + rg.off) + 2 * i;
      h2[0] = __floats2half2_rn(p.x, p.y); h2[1] = __floats2half2_rn(p.z, p.w);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (hp.shared_t) fs.iterations += 1; else fs.it_net[net] += 1;
    fs.rng_step += 1;
  }
}

// fp16 operand copy of a contiguous float range of the arena (f16 mode: uploaded parameters, test inputs)
__global__ void __launch_bounds__(256) k_to_half(const float* __restrict__ src, size_t n, OperandMode om) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    om.hbase[src + i - om.fbase] = __float2half_rn(src[i]);
}

// standalone flat Adam on caller-provided buffers (mrgan_adam_flat; unit tests + roofline probe)
__global__ void __launch_bounds__(256)
k_adam_plain(float4* __restrict__ p4, float4* __restrict__ m4, float4* __restrict__ v4, const float4* __restrict__ g4,
             long long n4, float lr_t, float b1, float b2, float eps) {
  const float c1 = 1.0f - b1, c2 = 1.0f - b2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 p = p4[i], m = m4[i], v = v4[i];
    const float4 g = __ldg(g4 + i);
#define ADAM1(c) m.c = fmaf(b1, m.c, c1 * g.c); v.c = fmaf(b2, v.c, c2 * g.c * g.c); p.c -= lr_t * m.c / (sqrtf(v.c) + eps);
    ADAM1(x) ADAM1(y) ADAM1(z) ADAM1(w)
#undef ADAM1
    p4[i] = p; m4[i] = m; v4[i] = v;
  }
}

// debug / test utility: materialise a block of the noise stream
__global__ void k_fill_normal(float* __restrict__ dst, const FoldState* __restrict__ folds, int fold, int step, int tid,
                              int rows, int cols, int row0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int r = i / cols, c = i % cols;
  const FoldState& fs = folds[fold];
  dst[i] = normal1(fs.key0, fs.key1, (uint32_t)(row0 + r), (uint32_t)c, (uint32_t)step, (uint32_t)tid);
}


// ------------------------------------------------------------------ device-side epoch permutations (mr_gan.py:189-202)
// The three index streams of an epoch, drawn on the device from a seed instead of being uploaded (3 x int32[n_train] per
// fold and epoch).  Stream 0 = labeled rows: floor(N / L) independent permutations of the L labeled rows followed by a
// permutation of the FIRST N mod L of them (mr_gan.py:189); streams 1 and 2 = permutations of all N training rows, or of
// the unlabeled subset tiled the same way (mr_gan.py:193-194,197-200).  A permutation of n items = the order of the keys
// (philox(i, tile, epoch, 0x50 + stream).x << 32) | i, sorted ascending (bitonic network in shared memory): unique keys,
// so the result is defined exactly and the oracle restates it with a stable argsort (oracle/fold_loop.py:device_perm).
struct PermDesc { const int* lab_rows; const int* unl_rows; int* idx; int n_lab, n_unl, n_train; uint32_t key0, key1; };

#define PERM_MAX 8192       // largest tile (64 KB of 64-bit keys)
__global__ void __launch_bounds__(1024)
k_epoch_perm(const PermDesc* __restrict__ descs, uint32_t epoch) {
  extern __shared__ unsigned long long pkeys[];
  const PermDesc d = descs[blockIdx.y];
  const int s = blockIdx.x;
  const int* const src = (s == 0) ? d.lab_rows : d.unl_rows;           // null: the rows themselves
  const int L = (s == 0) ? d.n_lab : (d.unl_rows ? d.n_unl : d.n_train);
  int* const out = d.idx + (size_t)s * d.n_train;
  const int N = d.n_train, ntiles = N / L, rem = N - ntiles * L;
  for (int j = 0; j <= ntiles; ++j) {
    const int n = (j < ntiles) ? L : rem;
    if (n == 0) break;
    int P = 1;
    while (P < n) P <<= 1;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
      unsigned long long k = ~0ull;
      if (i < n) k = ((unsigned long long)philox4x32_10(make_uint4((uint32_t)i, (uint32_t)j, epoch, 0x50u + (uint32_t)s), d.key0, d.key1).x << 32) | (uint32_t)i;
      pkeys[i] = k;
    }
    __syncthreads();
    for (int k2 = 2; k2 <= P; k2 <<= 1)
      for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
        for (int i = threadIdx.x; i < P; i += blockDim.x) {
          const int ixj = i ^ j2;
          if (ixj > i) {
            const unsigned long long a = pkeys[i], b = pkeys[ixj];
            const bool up = (i & k2) == 0;
            if ((a > b) == up) { pkeys[i] = b; pkeys[ixj] = a; }
          }
        }
        __syncthreads();
      }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int p = (int)(pkeys[i] & 0xffffffffull);
      out[(size_t)j * L + i] = src ? src[p] : p;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ device-side fold preparation (mr_gan.py:96-101)
// StandardScaler.fit over the training rows of a fold: per-column sum and sum of squares in float64.  Each of the
// gridDim.y row slices writes its own partial sums ([slice][2 * D]); the consumer adds the slices in slice order, so the
// statistics are bit-identical from run to run and whatever else shares the GPU (no floating-point atomics).
#define PREP_SLICES 64
__global__ void __launch_bounds__(128)
k_col_stats(const float* __restrict__ X, int ldx, const int* __restrict__ rows, int n_rows, int D, double* __restrict__ partials) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c >= D) return;
  double s = 0.0, q = 0.0;
  for (int i = blockIdx.y; i < n_rows; i += gridDim.y) {
    const double x = (double)X[(size_t)rows[i] * ldx + c];
    s += x; q += x * x;
  }
  partials[(size_t)blockIdx.y * 2 * D + c] = s;
  partials[(size_t)blockIdx.y * 2 * D + D + c] = q;
}

// StandardScaler.transform + row gather: out[i, c] = float((X[rows[i], c] - mean_c) / std_c), std 0 -> 1 (sklearn).
__global__ void __launch_bounds__(128)
k_scale_gather(const float* __restrict__ X, int ldx, const int* __restrict__ rows, int n_rows, int D, const double* __restrict__ partials,
               int n_slices, int n_fit, float* __restrict__ out, int ldo, const int* __restrict__ y_src, int* __restrict__ y_out, OperandMode om) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c >= D) return;
  double sum = 0.0, sq = 0.0;
  for (int sl = 0; sl < n_slices; ++sl) { sum += partials[(size_t)sl * 2 * D + c]; sq += partials[(size_t)sl * 2 * D + D + c]; }
  const double mean = sum / n_fit;
  double var = sq / n_fit - mean * mean;
  if (var < 0.0) var = 0.0;
  double sd = sqrt(var);
  if (sd < 1e-300 || var <= 10.0 * 2.220446049250313e-16 * fabs(mean) * fabs(mean)) sd = 1.0;   // constant column
  for (int i = blockIdx.y; i < n_rows; i += gridDim.y) {
    const float v = (float)(((double)X[(size_t)rows[i] * ldx + c] - mean) / sd);
    out[(size_t)i * ldo + c] = (om.mode == 1) ? rna_tf32(v) : v;
    if (om.mode == 2) om.hbase[out + (size_t)i * ldo + c - om.fbase] = __float2half_rn(v);     // X_test is a GEMM operand
    if (c == 0 && y_out) y_out[i] = y_src[rows[i]];
  }
}
