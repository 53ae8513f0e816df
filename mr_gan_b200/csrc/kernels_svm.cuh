// kernels_svm.cuh -- the RBF C-SVC of mr_svm.py:106 (sklearn's libsvm SVC(kernel='rbf', C)) for a group of folds.
//
// Specification: the libsvm source shipped with sklearn, sklearn/svm/src/libsvm/svm.cpp (cited as svm.cpp:<line>).
//   k_svm_split  tf32 hi / lo parts of every labeled and test row, and their row norms
//   k_svm_kmat   kernel matrices on tcgen05 (labeled x labeled, test x labeled), RBF transform in the epilogue
//   k_svm_smo    Solver::Solve without shrinking, one CTA per problem (fold, class pair; for mrgan_svm_cv also C and inner
//                split), alpha / G in double in shared memory
//   k_svm_vote   svm_predict_values' one-vs-one decision values and vote; k_svm_count the error count of a row set
#pragma once
#include "kernels_tc.cuh"

// ---------------------------------------------------------------- operands of the kernel matrix
// x = hi + lo + O(2^-22 |x|) with hi, lo on the tf32 grid (kind::tf32 MMAs read them without truncation).
// a.b ~ hi.hi + hi.lo + lo.hi: a 1-pass tf32 product is off by ~1e-5 in K, this 3-term split by ~1e-8.
struct SvmSplitOp {
  const float* X; int ldx;          // scaled rows (resident X_train / X_test)
  const int* rows;                  // rows of X to take (labeled rows), or nullptr: rows 0..n-1
  int n, D, Kp;                     // rows, features, padded features (multiple of 32)
  float *H, *L;                     // [n][Kp]
  double* norm;                     // [n]: sum hi^2 + 2 hi lo, the three terms of the GEMM (in double)
};

// one warp per row; blockIdx.y = op
__global__ void __launch_bounds__(256) k_svm_split(const SvmSplitOp* __restrict__ ops) {
  const SvmSplitOp op = ops[blockIdx.y];
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= op.n) return;
  const float* x = op.X + (size_t)(op.rows ? op.rows[r] : r) * op.ldx;
  float* H = op.H + (size_t)r * op.Kp;
  float* L = op.L + (size_t)r * op.Kp;
  double s = 0.0;
  for (int c = lane; c < op.Kp; c += 32) {
    const float v = c < op.D ? x[c] : 0.0f;
    const float hi = rna_tf32(v), lo = rna_tf32(v - hi);
    H[c] = hi; L[c] = lo;
    s += (double)hi * hi + 2.0 * ((double)hi * lo);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) op.norm[r] = s;
}

// ---------------------------------------------------------------- kernel matrix on tcgen05
// C[i][j] = exp(-gamma (|a_i|^2 + |b_j|^2 - 2 a_i.b_j)), b = labeled rows, a = labeled (ALAB) or test rows.
// MMA-M = 128 labeled rows b_j (TMEM lanes, so a warp stores 32 consecutive j: coalesced), MMA-N = 64 rows a_i.
// The contraction is dealt round-robin by 32-element k-block over SVM_NACC accumulators that the epilogue adds in double:
// each fp32 accumulator then sums 1/8 of the products, which keeps its rounding ~8x below one accumulator's
// (|a.b| reaches |a|^2 ~ D for similar rows).
#define SVM_BM 128
#define SVM_BN 64
#define SVM_NACC 8                                     // SVM_NACC x SVM_BN = 512 TMEM columns
#define SVM_STAGES 4
#define SVM_STAGE_BYTES (2 * SVM_BM * 128 + 2 * SVM_BN * 128)
#define SVM_KMAT_SMEM (1024 + SVM_STAGES * SVM_STAGE_BYTES + 256)
#define SVM_KMAT_THREADS (64 + 128)

struct alignas(64) SvmGemmOp {
  CUtensorMap mapBh, mapBl;         // labeled rows hi / lo: [nB][Kp] K-major, boxes of 32 x 128
  CUtensorMap mapAh, mapAl;         // row set a hi / lo:    [nA][Kp] K-major, boxes of 32 x 64
  const double *normA, *normB;
  float* C; int ldc;                // C[i * ldc + j]
  int nA, nB, Kp;
  float gamma;
  int same;                         // a == b (labeled x labeled): K(b_j, b_j) = 1 exactly, as libsvm computes it
};

__global__ void __launch_bounds__(SVM_KMAT_THREADS, 1) k_svm_kmat(const SvmGemmOp* __restrict__ ops) {
  using namespace tc;
  const SvmGemmOp& op = ops[blockIdx.z];
  const int j0 = blockIdx.x * SVM_BM, i0 = blockIdx.y * SVM_BN;
  if (j0 >= op.nB || i0 >= op.nA) return;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SVM_STAGES * SVM_STAGE_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + SVM_STAGES;
  uint64_t* tmem_full = bars + 2 * SVM_STAGES;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * SVM_STAGES + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = op.Kp / 32;
  if (warp == 0 && lane == 0) {
    prefetch_map(&op.mapBh); prefetch_map(&op.mapBl); prefetch_map(&op.mapAh); prefetch_map(&op.mapAl);
    for (int s = 0; s < SVM_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = *tmem_holder;
  constexpr uint32_t BBYTES = SVM_BM * 128, ABYTES = SVM_BN * 128;

  if (warp == 0) {
    if (lane == 0) {                                   // TMA producer
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % SVM_STAGES;
        mbar_wait(&empty[s], ((uint32_t)(kb / SVM_STAGES) & 1u) ^ 1u);
        mbar_expect_tx(&full[s], SVM_STAGE_BYTES);
        uint8_t* st = smem + (size_t)s * SVM_STAGE_BYTES;
        tma_load_2d(&op.mapBh, &full[s], st, kb * 32, j0);
        tma_load_2d(&op.mapBl, &full[s], st + BBYTES, kb * 32, j0);
        tma_load_2d(&op.mapAh, &full[s], st + 2 * BBYTES, kb * 32, i0);
        tma_load_2d(&op.mapAl, &full[s], st + 2 * BBYTES + ABYTES, kb * 32, i0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {                                   // MMA issuer: both operands K-major tf32, SWIZZLE_128B
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(SVM_BN >> 3) << 17) | ((uint32_t)(SVM_BM >> 4) << 24);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % SVM_STAGES;
        mbar_wait(&full[s], (uint32_t)(kb / SVM_STAGES) & 1u);
        fence_after();
        const uint32_t bh = smem_u32(smem + (size_t)s * SVM_STAGE_BYTES), bl = bh + BBYTES, ah = bh + 2 * BBYTES, al = ah + ABYTES;
        const uint32_t acc = tmem_base + (uint32_t)(SVM_BN * (kb % SVM_NACC));
#pragma unroll
        for (int k = 0; k < 4; ++k) {                  // 8 tf32 elements = 32 bytes per MMA
          const uint32_t first = (kb < SVM_NACC && k == 0) ? 0u : 1u;
          mma_tf32(acc, smem_desc(bh + 32 * k, 16, 1024, 2), smem_desc(ah + 32 * k, 16, 1024, 2), idesc, first);
          mma_tf32(acc, smem_desc(bh + 32 * k, 16, 1024, 2), smem_desc(al + 32 * k, 16, 1024, 2), idesc, 1u);
          mma_tf32(acc, smem_desc(bl + 32 * k, 16, 1024, 2), smem_desc(ah + 32 * k, 16, 1024, 2), idesc, 1u);
        }
        mma_commit(&empty[s]);
      }
      mma_commit(tmem_full);
    }
  } else {                                             // epilogue: thread = labeled row j, 16 rows i per TMEM load
    const int lane_base = 32 * (warp & 3);
    const int j = j0 + lane_base + lane;
    const bool j_ok = j < op.nB;
    const double nb = j_ok ? op.normB[j] : 0.0;
    const double g = (double)op.gamma;
    const int nacc = min(nkb, SVM_NACC);
    const int ncols = min(SVM_BN, op.nA - i0);
    mbar_wait(tmem_full, 0);
    fence_after();
    for (int c0 = 0; c0 < ncols; c0 += 16) {
      double s[16];
#pragma unroll
      for (int q = 0; q < 16; ++q) s[q] = 0.0;
      for (int a = 0; a < nacc; ++a) {
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)(SVM_BN * a + c0), v);
#pragma unroll
        for (int q = 0; q < 16; ++q) s[q] += (double)v[q];
      }
      if (j_ok) {
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const int i = i0 + c0 + q;
          if (i < op.nA) {
            const double d = fmax(op.normA[i] + nb - 2.0 * s[q], 0.0);
            op.C[(size_t)i * op.ldc + j] = (op.same && i == j) ? 1.0f : (float)exp(-g * d);
          }
        }
      }
    }
  }
  fence_before();
  __syncthreads();
  if (warp == 1) {
    fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------- batched SMO
#define SVM_SMO_THREADS 512
#define SVM_MAX_PAIR 8192                              // rows of one class pair: 24 bytes each in shared memory
#define SVM_SMO_SMEM_PER_ROW 24                        // alpha, G (double), QD (float), row map (int)
#define SVM_PER (SVM_MAX_PAIR / SVM_SMO_THREADS)
#define SVM_TAU 1e-12                                  // svm.cpp:105

struct SvmPairJob {
  const float* K; int ld;           // the fold's labeled x labeled matrix
  int a_off, na, b_off, nb;         // rows of class a (y = +1) and b (y = -1) in the labeled set (a_off / b_off: no row map)
  const int* rows;                  // [na + nb] row map into the labeled set (the class-a rows, then the class-b rows), or
                                    // nullptr: the contiguous segments a_off.. and b_off.. (mrgan_svm_fit)
  double C;                         // box constraint of this problem
  int ca, cb;                       // the two classes
  double* coef;                     // [na + nb]: alpha_k y_k (sv_coef)
  double* rho;
  int* n_iter; int* capped;
};

__device__ __forceinline__ int svm_row(const SvmPairJob& jb, int k) {
  return jb.rows ? jb.rows[k] : k < jb.na ? jb.a_off + k : jb.b_off + (k - jb.na);
}

// (value, index) arg-max with libsvm's scan order: on equal values the larger index wins (svm.cpp:964,973 use >=)
__device__ __forceinline__ void svm_max_last(double& v, int& i, double v2, int i2) {
  if (v2 > v || (v2 == v && i2 > i)) { v = v2; i = i2; }
}
// arg-min, on equal values the larger index wins (svm.cpp:1003,1027 use <=)
__device__ __forceinline__ void svm_min_last(double& v, int& i, double v2, int i2) {
  if (v2 < v || (v2 == v && i2 > i)) { v = v2; i = i2; }
}

// Solver::Solve (svm.cpp:666-943) for the C-SVC sub-problem of one class pair, no shrinking.  The reductions combine
// (value, index) with a total order, so the result does not depend on the reduction tree: bitwise reproducible.
// Double arithmetic is written with _rn intrinsics so that no product is contracted into an FMA (libsvm's host build
// rounds every product).
// The row map is read once into shared memory, so the scans below load only K from global memory.
__global__ void __launch_bounds__(SVM_SMO_THREADS) k_svm_smo(const SvmPairJob* __restrict__ jobs, double eps) {
  const SvmPairJob jb = jobs[blockIdx.x];
  const int n = jb.na + jb.nb;
  const double C = jb.C;
  extern __shared__ double svm_smem[];
  double* alpha = svm_smem;                            // [n]
  double* G = alpha + n;                               // [n]
  float* QD = reinterpret_cast<float*>(G + n);         // [n]: K(k, k)
  int* row = reinterpret_cast<int*>(QD + n);           // [n]: row of problem row k in the labeled set
  __shared__ double r1v[SVM_SMO_THREADS / 32], r2v[SVM_SMO_THREADS / 32], r2m[SVM_SMO_THREADS / 32];
  __shared__ int r1i[SVM_SMO_THREADS / 32], r2i[SVM_SMO_THREADS / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int NW = SVM_SMO_THREADS / 32;
  for (int k = tid; k < n; k += SVM_SMO_THREADS) {
    alpha[k] = 0.0; G[k] = -1.0;                       // alpha = 0, G = p = -1 (svm.cpp:703)
    const int r = svm_row(jb, k);
    row[k] = r;
    QD[k] = jb.K[(size_t)r * jb.ld + r];
  }
  __syncthreads();
  const long long cap = max(10000000LL, 100LL * n);
  long long iter = 0;
  int capped = 0;
  float qi[SVM_PER];
  while (true) {
    if (iter >= cap) { capped = 1; break; }
    // ---- i = argmax over I_up of -y_t G_t (svm.cpp:960-978)
    double gv = -INFINITY; int gi = -1;
#pragma unroll
    for (int s = 0; s < SVM_PER; ++s) {
      const int k = tid + s * SVM_SMO_THREADS;
      if (k >= n) break;
      const double a = alpha[k], yk = k < jb.na ? 1.0 : -1.0;
      if (yk > 0 ? a < C : a > 0.0) svm_max_last(gv, gi, -yk * G[k], k);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) svm_max_last(gv, gi, __shfl_xor_sync(0xffffffffu, gv, o), __shfl_xor_sync(0xffffffffu, gi, o));
    if (lane == 0) { r1v[warp] = gv; r1i[warp] = gi; }
    __syncthreads();
    double Gmax = -INFINITY; int i = -1;
    for (int w = 0; w < NW; ++w) svm_max_last(Gmax, i, r1v[w], r1i[w]);
    // ---- j: second-order rule over I_low (svm.cpp:985-1035)
    double g2 = -INFINITY, om = INFINITY; int oj = -1;
    const double yi = i < jb.na ? 1.0 : -1.0;
    const float* Ki = jb.K + (size_t)row[i >= 0 ? i : 0] * jb.ld;
    const double QDi = i >= 0 ? (double)QD[i] : 0.0;
#pragma unroll
    for (int s = 0; s < SVM_PER; ++s) {
      const int k = tid + s * SVM_SMO_THREADS;
      if (k >= n) break;
      qi[s] = i >= 0 ? Ki[row[k]] : 0.0f;
      const double a = alpha[k], yk = k < jb.na ? 1.0 : -1.0;
      if (yk > 0 ? a > 0.0 : a < C) {
        const double yG = yk * G[k];
        g2 = fmax(g2, yG);
        const double gd = __dadd_rn(Gmax, yG);
        if (i >= 0 && gd > 0) {
          double quad = __dsub_rn(__dadd_rn(QDi, (double)QD[k]), __dmul_rn(2.0, (double)qi[s]));   // QD_i + QD_j - 2 K_ij
          if (!(quad > 0)) quad = SVM_TAU;
          svm_min_last(om, oj, -__ddiv_rn(__dmul_rn(gd, gd), quad), k);
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      g2 = fmax(g2, __shfl_xor_sync(0xffffffffu, g2, o));
      svm_min_last(om, oj, __shfl_xor_sync(0xffffffffu, om, o), __shfl_xor_sync(0xffffffffu, oj, o));
    }
    if (lane == 0) { r2v[warp] = g2; r2m[warp] = om; r2i[warp] = oj; }
    __syncthreads();
    double Gmax2 = -INFINITY, omin = INFINITY; int j = -1;
    for (int w = 0; w < NW; ++w) { Gmax2 = fmax(Gmax2, r2v[w]); svm_min_last(omin, j, r2m[w], r2i[w]); }
    if (Gmax + Gmax2 < eps || j == -1) break;          // svm.cpp:1037
    ++iter;
    // ---- two-variable update with box clipping (svm.cpp:761-855); every thread computes it, identically
    const double yj = j < jb.na ? 1.0 : -1.0;
    const double Kij = (double)Ki[row[j]], QDj = (double)QD[j];
    const double ai = alpha[i], aj = alpha[j], Gi = G[i], Gj = G[j];
    double ni, nj;
    if (yi != yj) {
      double quad = __dadd_rn(__dadd_rn(QDi, QDj), __dmul_rn(2.0, -Kij));   // Q_ij = -K_ij
      if (quad <= 0) quad = SVM_TAU;
      const double delta = __ddiv_rn(__dsub_rn(-Gi, Gj), quad);
      const double diff = __dsub_rn(ai, aj);
      ni = __dadd_rn(ai, delta); nj = __dadd_rn(aj, delta);
      if (diff > 0) { if (nj < 0) { nj = 0; ni = diff; } }
      else { if (ni < 0) { ni = 0; nj = -diff; } }
      if (diff > 0) { if (ni > C) { ni = C; nj = __dsub_rn(C, diff); } }   // C_i - C_j = 0
      else { if (nj > C) { nj = C; ni = __dadd_rn(C, diff); } }
    } else {
      double quad = __dsub_rn(__dadd_rn(QDi, QDj), __dmul_rn(2.0, Kij));   // Q_ij = K_ij
      if (quad <= 0) quad = SVM_TAU;
      const double delta = __ddiv_rn(__dsub_rn(Gi, Gj), quad);
      const double sum = __dadd_rn(ai, aj);
      ni = __dsub_rn(ai, delta); nj = __dadd_rn(aj, delta);
      if (sum > C) { if (ni > C) { ni = C; nj = __dsub_rn(sum, C); } }
      else { if (nj < 0) { nj = 0; ni = sum; } }
      if (sum > C) { if (nj > C) { nj = C; ni = __dsub_rn(sum, C); } }
      else { if (ni < 0) { ni = 0; nj = sum; } }
    }
    const double dai = __dsub_rn(ni, ai), daj = __dsub_rn(nj, aj);
    const float* Kj = jb.K + (size_t)row[j] * jb.ld;
    __syncthreads();                                   // everybody has read alpha / G of i and j
    if (tid == 0) { alpha[i] = ni; alpha[j] = nj; }
#pragma unroll
    for (int s = 0; s < SVM_PER; ++s) {                // G_k += Q_ik dai + Q_jk daj (svm.cpp:862-865)
      const int k = tid + s * SVM_SMO_THREADS;
      if (k >= n) break;
      const double yk = k < jb.na ? 1.0 : -1.0;
      const double Qik = yi * yk * (double)qi[s], Qjk = yj * yk * (double)Kj[row[k]];
      G[k] = __dadd_rn(G[k], __dadd_rn(__dmul_rn(Qik, dai), __dmul_rn(Qjk, daj)));
    }
    __syncthreads();                                   // alpha[i], alpha[j] visible to the owners' next scan
  }
  __syncthreads();
  for (int k = tid; k < n; k += SVM_SMO_THREADS) jb.coef[k] = k < jb.na ? alpha[k] : -alpha[k];
  if (tid == 0) {                                      // calculate_rho, svm.cpp:1126-1162, in libsvm's order
    double ub = INFINITY, lb = -INFINITY, sum_free = 0.0;
    int nr_free = 0;
    for (int k = 0; k < n; ++k) {
      const double yk = k < jb.na ? 1.0 : -1.0, yG = yk * G[k], a = alpha[k];
      if (a >= C) { if (yk < 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
      else if (a <= 0) { if (yk > 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
      else { ++nr_free; sum_free = __dadd_rn(sum_free, yG); }
    }
    *jb.rho = nr_free > 0 ? sum_free / nr_free : (ub + lb) / 2;
    *jb.n_iter = (int)iter;
    *jb.capped = capped;
  }
}

// ---------------------------------------------------------------- decision values and vote (svm.cpp:2865-2897)
#define SVM_VOTE_THREADS 256
// one CTA per (row t, row set f): the models of set f are jobs[f * npairs ...]; Kt[f] = its rows x labeled kernel matrix,
// whose row t is the voted row, or row trow[f][t] when trow is given (the validation rows of mrgan_svm_cv's inner splits,
// rows of the labeled x labeled matrix).  dec_out, wrong (with yte) and pred may be null: rows without labels
// (mrgan_predict_rows) store only the voted class, the validation rows only their wrong flags.
__global__ void __launch_bounds__(SVM_VOTE_THREADS) k_svm_vote(const SvmPairJob* __restrict__ jobs, int npairs, int n_classes,
                                                               const float* const* __restrict__ Kt, const int* const* __restrict__ trow,
                                                               const int* const* __restrict__ yte, const int* __restrict__ n_test,
                                                               float* const* __restrict__ dec_out, int* const* __restrict__ wrong,
                                                               int* const* __restrict__ pred) {
  const int f = blockIdx.y, t = blockIdx.x;
  if (t >= n_test[f]) return;
  const SvmPairJob* jf = jobs + (size_t)f * npairs;
  const int ld = jf[0].ld;
  const float* row = Kt[f] + (size_t)(trow ? trow[f][t] : t) * ld;
  __shared__ float dec_s[2048];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int p = warp; p < npairs; p += SVM_VOTE_THREADS / 32) {
    const SvmPairJob& jb = jf[p];
    const int n = jb.na + jb.nb;
    double s = 0.0;
    for (int k = lane; k < n; k += 32) s = __dadd_rn(s, __dmul_rn(jb.coef[k], (double)row[svm_row(jb, k)]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
    if (lane == 0) {
      const double d = s - *jb.rho;
      if (dec_out) dec_out[f][(size_t)t * npairs + p] = (float)d;
      dec_s[p] = d > 0 ? 1.0f : 0.0f;                  // the vote only needs the sign
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int votes[64];
    for (int c = 0; c < n_classes; ++c) votes[c] = 0;
    for (int p = 0; p < npairs; ++p) ++votes[dec_s[p] > 0.5f ? jf[p].ca : jf[p].cb];
    int best = 0;
    for (int c = 1; c < n_classes; ++c) if (votes[c] > votes[best]) best = c;   // the first class with most votes
    if (wrong) wrong[f][t] = best != yte[f][t];
    if (pred) pred[f][t] = best;
  }
}

// error count of each row set (blockIdx.x: a fold's test rows, or a validation split), summed in a fixed order
__global__ void __launch_bounds__(256) k_svm_count(int* const* __restrict__ wrong, const int* __restrict__ n_test, int* __restrict__ count) {
  const int f = blockIdx.x, n = n_test[f];
  __shared__ int part[256];
  int s = 0;
  for (int t = threadIdx.x; t < n; t += 256) s += wrong[f][t];
  part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int c = 0;
    for (int w = 0; w < 256; ++w) c += part[w];
    count[f] = c;
  }
}
