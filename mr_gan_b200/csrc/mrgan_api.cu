// mrgan_api.cu -- handle, memory layout, launch sequences, CUDA-graph epoch and the C-ABI
// declared in include/mrgan.h.  Reference interface replaced: the K.function callables of
// mr_gan.py:169-171, the epoch loop mr_gan.py:183-230 and mr_nn.py:114-118.
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/mrgan.h"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_svm.cuh"
#include "kernels_dp.cuh"

namespace {

thread_local std::string g_last_error;

// ------------------------------------------------------------------ op table
enum Op {
  OP_G1, OP_G2, OP_G3D, OP_G3G,
  OP_D1, OP_D2, OP_D3, OP_D4, OP_D5, OP_D6,
  OP_DW1, OP_DW2, OP_DW3, OP_DW4, OP_DW5, OP_DW6,
  OP_DX2, OP_DX3, OP_DX4, OP_DX5, OP_DX6,     // OP_DXl: dZ[l] -> dZ[l-1]
  OP_DX1G,                                     // dZ[1] -> dFake (G step only)
  OP_D1G, OP_D2G, OP_D3G, OP_D4G, OP_D5G,      // G step: D forward over 2B rows [fake | real] (own TMA boxes / MMA-N)
  OP_DX2G, OP_DX3G, OP_DX4G, OP_DX5G,          // G step: dX chain over the B fake rows
  OP_GW1, OP_GW2, OP_GW3, OP_GX2, OP_GX3,
  OP_E1, OP_E1S, OP_E2, OP_E3, OP_E4, OP_E5, OP_E6,
  NUM_OPS,
  // eval backward (mrgan_input_grad / mrgan_saliency), the twins of OP_DX2..6 / OP_DX1G over the phase-0 activations.  Their
  // device descriptors live in a workspace made on first use (SalWork), outside the arena's [NUM_OPS][nf] table.
  OP_EX2 = NUM_OPS, OP_EX3, OP_EX4, OP_EX5, OP_EX6,   // OP_EXl: dZ[l] -> dZ[l-1], written over eh[l-1]
  OP_EX1,                                            // dZ[1] -> d/dx, fp32 into ex_stage
  // samples of the generator (mrgan_generate / mrgan_sample_stats), over up to NG = batch * floor(NE / batch) rows per fold;
  // device descriptors in the workspace GenWork.  OP_GGl: twins of OP_G1, OP_G2, OP_G3G (no noise: OP_GG3 writes the clean rows
  // and their operand copy into ex_stage); OP_Sl: D's eval forward over those staged rows (twins of OP_E1S, OP_E2 .. OP_E6)
  OP_GG1, OP_GG2, OP_GG3,
  OP_S1, OP_S2, OP_S3, OP_S4, OP_S5, OP_S6,
  NUM_OPS_ALL
};
constexpr int NUM_EX = OP_GG1 - NUM_OPS;
constexpr int NUM_GEN = NUM_OPS_ALL - OP_GG1;

struct OpInfo { bool at = false, bt = false, used = false; int maxM = 0, maxN = 0; };

// How a tcgen05 op is launched: decided once per handle by tc_plan_op, read by tc_launch_gemm.
struct TcKernel;
struct TcPlan {
  const TcKernel* k = nullptr;   // the k_gemm_tc instantiation (tc_kernel); null for an unused op or a fused one
  bool fused = false;            // dW runs fused with Adam in k_dw_adam_tc (tc_launch_dw_adam)
  int gx = 0;                    // grid.x: feature tiles
  int bn = 0;                    // batch rows per tile, the most of any fold (grid.y)
  int bn_big = 256;              // batch rows per tile of a fold with more than 256 rows (forward / dX)
  int maxME = 0, maxNE = 0;      // extents over the folds: MMA-M (features), MMA-N (batch rows)
  size_t smem = 0;               // dynamic shared memory of a launch
  int ks = 1;                    // contraction slices per tile (deterministic split-K of a large-batch dW)
};

struct Arena {
  char* base = nullptr; size_t off = 0;
  template <typename T> T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

struct TensorLayout { int rows, cols, pitch; long long off; };   // inside a net's flat block

struct NetLayout {
  std::vector<TensorLayout> t;   // D: 6 augmented matrices; G: W1aug, gamma, beta, W2aug, W3aug
  long long n = 0;               // padded length (multiple of 32)
  long long n_ref = 0;           // length in the reference's packed order
  long long off = 0;             // offset of this net in the handle's flat buffers
};

struct FoldBuffers {
  float *a[6], *hb[6], *dz[6], *lg, *dlg, *dfake, *zb, *h1g, *xhat, *istd, *u, *h2g, *dz2g, *du, *dz1g;
  float *stage_x, *stage_z, *ex_stage, *xte, *eh[6], *elg, *xtr, *eval_out, *eval_out_s;
  int *stage_y, *labels_cur, *ey_stage, *ytr, *yte, *idx;
  int *pred, *pred_s;            // predicted classes of the resident test set / of the staged rows (mrgan_predict*)
  int *lab_rows, *unl_rows;      // device-side epoch permutations: labeled / unlabeled row subsets (mrgan_set_epoch_rows)
  int n_lab = 0, n_unl = 0;
  int lda[6], ldz[6];   // pitches of a/h (with ones column) and dz
  bool loaded = false;
};

}  // namespace

struct mrgan_handle;
namespace {
int tc_setup(mrgan_handle* h);
int tc_views(mrgan_handle* h, int op0, int op1, TcOp* dst);
void tc_teardown(mrgan_handle* h);
void tc_launch_gemm(mrgan_handle* h, int op, int f0, int nfl, int rows_override, cudaStream_t st, const OperandMode& om);
void tc_launch_dw_adam(mrgan_handle* h, int op, int nlayers, int f0, int nfl, cudaStream_t st);
int tc_debug_gemm(mrgan_handle* h, int mode, const GemmDesc& g, int esz);
}

constexpr int kMaxChains = 16;
struct mrgan_handle {
  mrgan_config cfg;
  int nf = 0, R = 0, NE = 0, n_train = 0;
  std::vector<mrgan_fold_shape> shapes;
  std::vector<NetLayout> net[2];
  std::vector<FoldBuffers> fb;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;        // dW (+Adam) kernels run here, concurrently with the latency-bound dX chain
  cudaEvent_t ev_pool[16] = {nullptr}; int ev_next = 0;
  bool side_open = false;             // work forked to `side` since the last join (joins are no-ops otherwise)
  // the folds of a group are independent, so an epoch is captured as `nchains` parallel chains of kernels (disjoint fold
  // ranges, own main + side stream): one chain's latency-bound small kernels fill the SMs another chain leaves idle
  int nchains = 1;
  cudaStream_t cmain[kMaxChains] = {nullptr}, cside[kMaxChains] = {nullptr};
  char* arena = nullptr; size_t arena_bytes = 0;
  __half* harena = nullptr;           // f16 mode: one __half per float of the arena (operand copies at the same element index)
  OperandMode om = {0, 1.0f, nullptr, nullptr};
  float *P = nullptr, *Mo = nullptr, *Vo = nullptr, *Gr = nullptr; long long n_flat = 0;
  FoldState* d_folds = nullptr; std::vector<FoldState> h_folds;
  GemmDesc* d_descs = nullptr; std::vector<GemmDesc> h_descs;
  PermDesc* d_perm = nullptr;
  BnDesc* d_bn = nullptr; LossDesc* d_loss = nullptr; EvalDesc *d_eval = nullptr, *d_eval_s = nullptr;
  int* d_conf = nullptr;              // [nf][K][K] confusion counts (mrgan_confusion)
  // mrgan_input_grad / mrgan_saliency: one allocation on first use (a handle that never calls them allocates nothing more)
  struct SalWork {
    char* mem = nullptr;
    GemmDesc* descs = nullptr;        // [NUM_EX][nf] device copies of the OP_EX* descriptors
    float* profile = nullptr;         // [nf][K][D_max]
    TcOp* tcops = nullptr;            // [NUM_EX][nf] their tcgen05 views (tf32 / f16 handles)
  } sal;
  // mrgan_generate / mrgan_sample_stats: the same pattern.  The generator's activations live here, the operand buffers (z, u,
  // h2) first, covered by the workspace's own fp16 shadow (f16 handles) and OperandMode; the eval buffers stay untouched
  // except ex_stage / eh / elg, whose contents are dead between calls.
  struct GenWork {
    char* mem = nullptr; __half* hmem = nullptr;
    OperandMode om = {0, 1.0f, nullptr, nullptr};   // fbase = mem, hbase = hmem
    size_t hfloats = 0;               // floats of mem with an fp16 copy
    int NG = 0, nseg = 0, ldz = 0;    // rows per chunk (whole batches), batch segments per chunk, pitch of z
    size_t zstride = 0;               // floats between the z buffers of consecutive folds
    float* z = nullptr;               // [nf][NG][ldz]
    float* zs = nullptr;              // [NG][noise_dim]: a chunk of the caller's z (mrgan_generate)
    GemmDesc* descs = nullptr;        // [NUM_GEN][nf]
    TcOp* tcops = nullptr;            // [NUM_GEN][nf] (tf32 / f16 handles)
    BnDesc* bn = nullptr;             // [nf][nseg]: BatchNorm of each batch segment
    StatsDesc* st = nullptr;          // [2][nf]: generated rows, resident test rows
    double *s1 = nullptr, *s2 = nullptr, *score = nullptr; int* counts = nullptr;   // [nf][2][SS_W], [nf][2][SS_W^2], [nf][2], [nf][64]
  } gen;
  AdamRange* d_ranges[2] = {nullptr, nullptr};
  OpInfo ops[NUM_OPS_ALL];
  float *d_step_stats = nullptr, *d_epoch_stats = nullptr, *h_epoch_stats = nullptr;
  int* h_idx_pinned[2] = {nullptr, nullptr}; cudaEvent_t idx_free[2] = {nullptr, nullptr}; int idx_slot = 0;
  float* h_scratch = nullptr;   // pinned scalars for the step API
  std::map<int, cudaGraphExec_t> graphs;   // key: nb (GAN) or n_idx (NN)
  std::map<int, long long> graph_nodes;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool epoch_pending = false; double last_ms = 0.0;
  long long launches = 0;
  std::string err;
  int sticky = 0;                     // first failure of a call that cannot return a status itself (kernel launch, NCCL enqueue):
                                      // surfaced by the next public entry point through take_sticky()
  AdamHyper hp;
  // data-parallel mode (mrgan_dp_init): NCCL communicator + buffers of the all-reduced batch statistics
  // device-resident raw datasets (mrgan_load_dataset) and scratch of the device-side fold preparation
  struct Dataset { float* x = nullptr; int* y = nullptr; int n = 0, D = 0, ld = 0; } datasets[8];
  double* d_prep_stats = nullptr; int* d_prep_rows = nullptr; int prep_rows_cap = 0, prep_stats_cap = 0;
  int dp_world = 1, dp_rank = 0;
  bool dp_virtual = false;            // the handle's folds play the ranks (mrgan_dp_init_virtual): collectives are local sums
  // fused gradient exchange (kernels_dp.cuh): peer mappings of every rank's arena (cudaIpc), flag blocks, per-net pointer sets
  bool dp_fused = false;
  unsigned* d_dpflags = nullptr;      // DP_MAX_RANKS x DP_FLAG_WORDS words inside the arena (zero at creation)
  char* peer_arena[DP_MAX_RANKS] = {nullptr}; __half* peer_harena[DP_MAX_RANKS] = {nullptr};
  DpPeers dp_peers[2];                // [net]
  void* nccl_comm = nullptr;
  float* d_dpmem = nullptr; DpBufs* d_dpbufs = nullptr;
  float *dp_bnf = nullptr, *dp_bnb = nullptr, *dp_fm = nullptr;   // [nf][2*500], [nf][2*500], [nf][2*250]
  float* dp_losspart = nullptr; unsigned* dp_lossctr = nullptr;    // k_loss_disc block partials [nf][4*64] and arrival counters [nf]
  TcOp* d_tcops = nullptr;            // [NUM_OPS][nf] tensor maps + epilogue descriptors
  TcPlan tc_plan[NUM_OPS_ALL];
  float* d_tcws = nullptr;            // partial products of the split-K dW ops
  bool tc_fused_adam = false;         // dW and Adam in one kernel, k_dw_adam_tc (no gradient round trip); tcgen05 handles only
  int tc_heads = 0;                   // losses / feature matching / BatchNorm fused into GEMM epilogues (set by tc_setup), bit mask:
                                      // 1 = HEAD_DISC (no k_loss_disc, no k_adam of D), 2 = HEAD_FM (no k_fm), 4 = HEAD_BN (no k_bn_fwd)
  TcAdamOp* d_tcadam = nullptr;       // [NUM_OPS][nf]
  AdamRange* d_ranges_tc[2] = {nullptr, nullptr};   // what is left for k_adam: BN gamma/beta (G), nothing (D)
  // MRGAN_MODEL_SVM: workspace of mrgan_svm_fit (one allocation, reused while it is large enough)
  struct Svm {
    char* mem = nullptr; size_t bytes = 0;
    int n_lab = 0, npairs = 0, npmax = 0, max_rows = 0, max_nte = 0;
    double eps = 1e-3;
    bool fitted = false;
    std::vector<float*> Klab, Kte, dec;
    std::vector<int*> wrong;
    int *d_iters = nullptr, *d_capped = nullptr, *d_count = nullptr, *d_nte = nullptr;
    SvmSplitOp* d_split = nullptr; SvmGemmOp* d_gemm = nullptr; SvmPairJob* d_jobs = nullptr;
    float** d_Kt = nullptr; float** d_dec = nullptr; int** d_yte = nullptr; int** d_wrong = nullptr; int** d_pred = nullptr;
    // mrgan_predict_rows: up to max_nte new rows of one fold, staged, split, kernel matrix, decision values and vote
    std::vector<SvmGemmOp> h_gemm;      // host copies of the descriptors in d_gemm
    float *Xs = nullptr, *Hs = nullptr, *Ls = nullptr, *Ks = nullptr, *decs = nullptr; double* ns = nullptr; int* preds = nullptr;
    SvmSplitOp* d_split_s = nullptr; SvmGemmOp* d_gemm_s = nullptr;
    float** d_Ks = nullptr; float** d_decs = nullptr; int** d_preds = nullptr; int* d_ns = nullptr;   // one-fold pointer tables
    // mrgan_svm_cv: problems, row maps, validation rows and counts of every (fold, C, inner split), beside the fit's workspace
    char* cv_mem = nullptr; size_t cv_bytes = 0;
  } svm;
};

namespace {

int take_sticky(mrgan_handle* h);

int fail(mrgan_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  g_last_error = msg;
  return code;
}

#define CKS()                                                                                      \
  do {                                                                                             \
    CK(cudaGetLastError());                                                                        \
    const int _s = take_sticky(h);                                                                 \
    if (_s) return _s;                                                                             \
  } while (0)

#define CK(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail(h, MRGAN_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
  } while (0)

const int kDW[5] = {1000, 500, 250, 250, 250};   // mr_gan.py:119-127
const int kGH = 500;                               // mr_gan.py:111,113

long long align32(long long x) { return (x + 31) & ~31LL; }

NetLayout layout_disc(int D, int K) {
  NetLayout L;
  int dims[7] = {D, kDW[0], kDW[1], kDW[2], kDW[3], kDW[4], K};
  for (int l = 0; l < 6; ++l) {
    TensorLayout t{dims[l] + 1, dims[l + 1], pitch8(dims[l + 1]), L.n};
    L.t.push_back(t);
    L.n = align32(L.n + (long long)t.rows * t.pitch);
    L.n_ref += (long long)(dims[l] + 1) * dims[l + 1];
  }
  return L;
}

NetLayout layout_gen(int D, int nd) {
  NetLayout L;
  auto add = [&](int rows, int cols) {
    TensorLayout t{rows, cols, pitch8(cols), L.n};
    L.t.push_back(t);
    L.n = align32(L.n + (long long)rows * t.pitch);
    L.n_ref += (long long)rows * cols;
  };
  add(nd + 1, kGH);   // W1aug
  add(1, kGH);        // gamma
  add(1, kGH);        // beta
  add(kGH + 1, kGH);  // W2aug
  add(kGH + 1, D);    // W3aug
  return L;
}

__global__ void k_round_tf32(float* p, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = rna_tf32(p[i]);
}

__global__ void k_set_col(float* p, int ld, int rows, int col, float v, OperandMode om) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows) {
    p[(size_t)r * ld + col] = v;
    if (om.mode == 2) om.hbase[p + (size_t)r * ld + col - om.fbase] = __float2half_rn(v);
  }
}

__global__ void k_scale_buf(float* p, size_t n, float mul) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] *= mul;
}

// f16 mode, test hook: operand-only buffers exist as fp16 copies only; expand one (times `mul`) into a float scratch
__global__ void k_from_half(const float* src, float* dst, size_t n, float mul, OperandMode om) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dst[i] = __half2float(om.hbase[src + i - om.fbase]) * mul;
}

// ---- buffer layout (run twice: sizing pass with base == nullptr, then for real) ----
void layout_buffers(mrgan_handle* h, Arena& ar) {
  const mrgan_config& c = h->cfg;
  const int B = c.batch, R = h->R, NE = h->NE, K = c.n_classes, nd = c.noise_dim, nf = h->nf;
  const bool gan = c.model == MRGAN_MODEL_GAN;
  if (c.model == MRGAN_MODEL_SVM) {     // fold data only (what mrgan_load_fold / mrgan_prepare_fold write)
    for (int f = 0; f < nf; ++f) {
      FoldBuffers& b = h->fb[f];
      const int D = h->shapes[f].D;
      b.lda[0] = pitch8(D + 1);
      b.xte = ar.take<float>((size_t)h->shapes[f].n_test * b.lda[0]);
      b.xtr = ar.take<float>((size_t)h->shapes[f].n_train * pitch8(D));
      b.ytr = ar.take<int>(h->shapes[f].n_train);
      b.yte = ar.take<int>(h->shapes[f].n_test);
      b.pred = ar.take<int>(h->shapes[f].n_test);
    }
    h->d_eval = ar.take<EvalDesc>(nf);
    h->d_conf = ar.take<int>((size_t)nf * K * K);
    return;
  }
  h->P = ar.take<float>(h->n_flat);
  h->Mo = ar.take<float>(h->n_flat);
  h->Vo = ar.take<float>(h->n_flat);
  h->Gr = ar.take<float>(h->n_flat);
  h->d_folds = ar.take<FoldState>(nf);
  h->d_descs = ar.take<GemmDesc>((size_t)NUM_OPS * nf);
  h->d_perm = ar.take<PermDesc>(nf);
  h->d_bn = ar.take<BnDesc>(nf);
  h->d_loss = ar.take<LossDesc>(nf);
  h->d_eval = ar.take<EvalDesc>(nf);
  h->d_eval_s = ar.take<EvalDesc>(nf);
  h->d_ranges[0] = ar.take<AdamRange>(nf);
  h->d_ranges[1] = ar.take<AdamRange>(nf);
  h->d_step_stats = ar.take<float>((size_t)(h->n_train / B + 1) * nf * 4);
  h->d_dpflags = ar.take<unsigned>((size_t)DP_MAX_RANKS * DP_FLAG_WORDS);
  h->d_epoch_stats = ar.take<float>((size_t)nf * 8);
  for (int f = 0; f < nf; ++f) {
    FoldBuffers& b = h->fb[f];
    const int D = h->shapes[f].D, ntr = h->shapes[f].n_train, nte = h->shapes[f].n_test;
    const int ldx = pitch8(D);
    int win[6] = {D, kDW[0], kDW[1], kDW[2], kDW[3], kDW[4]};
    for (int l = 0; l < 6; ++l) { b.lda[l] = pitch8(win[l] + 1); b.ldz[l] = pitch8(win[l]); }
    b.a[0] = ar.take<float>((size_t)R * b.lda[0]);
    b.hb[0] = nullptr; b.dz[0] = nullptr;
    for (int l = 1; l <= 5; ++l) {
      b.hb[l] = ar.take<float>((size_t)R * b.lda[l]);
      b.a[l] = (l < 5) ? ar.take<float>((size_t)R * b.lda[l]) : b.hb[l];
      b.dz[l] = ar.take<float>((size_t)R * b.ldz[l]);
    }
    b.lg = ar.take<float>((size_t)R * pitch8(K));
    b.dlg = ar.take<float>((size_t)R * pitch8(K));
    b.labels_cur = ar.take<int>(R);
    b.stage_x = ar.take<float>((size_t)R * ldx);
    b.stage_y = ar.take<int>(R);
    if (gan) {
      b.dfake = ar.take<float>((size_t)B * ldx);
      b.zb = ar.take<float>((size_t)B * pitch8(nd + 1));
      const int ldg = pitch8(kGH);
      b.h1g = ar.take<float>((size_t)B * ldg);
      b.xhat = ar.take<float>((size_t)B * ldg);
      b.istd = ar.take<float>(kGH);
      b.u = ar.take<float>((size_t)B * pitch8(kGH + 1));
      b.h2g = ar.take<float>((size_t)B * pitch8(kGH + 1));
      b.dz2g = ar.take<float>((size_t)B * ldg);
      b.du = ar.take<float>((size_t)B * ldg);
      b.dz1g = ar.take<float>((size_t)B * ldg);
      b.stage_z = ar.take<float>((size_t)B * nd);
    }
    b.ex_stage = ar.take<float>((size_t)NE * b.lda[0]);
    b.xte = ar.take<float>((size_t)nte * b.lda[0]);
    for (int l = 1; l <= 5; ++l) b.eh[l] = ar.take<float>((size_t)NE * b.lda[l]);
    b.elg = ar.take<float>((size_t)NE * pitch8(K));
    b.ey_stage = ar.take<int>(NE);
    b.eval_out = ar.take<float>(4);
    b.eval_out_s = ar.take<float>(4);
    b.xtr = ar.take<float>((size_t)ntr * ldx);
    b.ytr = ar.take<int>(ntr);
    b.yte = ar.take<int>(nte);
    b.idx = ar.take<int>((size_t)3 * ntr);
    b.lab_rows = ar.take<int>(ntr);
    b.unl_rows = ar.take<int>(ntr);
    b.pred = ar.take<int>(nte);
    b.pred_s = ar.take<int>(NE);
  }
  h->d_conf = ar.take<int>((size_t)nf * K * K);
}

GemmDesc make_desc(const float* A, int lda, const float* Bm, int ldb, float* C, int ldc, int M, int N, int K, int epi,
                   int act, int fold) {
  GemmDesc d;
  memset(&d, 0, sizeof(d));
  d.A = A; d.lda = lda; d.B = Bm; d.ldb = ldb; d.C = C; d.ldc = ldc; d.M = M; d.N = N; d.K = K;
  d.epi = epi; d.act = act; d.fold = fold;
  return d;
}

// the host descriptor of op for fold f; rnd: which outputs feed a tensor-core GEMM as operands (tf32 / f16 handles)
void set_op(mrgan_handle* h, int op, int f, GemmDesc d, bool at, bool bt, int rnd) {
  d.rnd = h->cfg.precision != MRGAN_PREC_FP32 ? rnd : 0;
  h->h_descs[(size_t)op * h->nf + f] = d;
  OpInfo& oi = h->ops[op];
  oi.at = at; oi.bt = bt; oi.used = true;
  if (d.M > oi.maxM) oi.maxM = d.M;
  if (d.N > oi.maxN) oi.maxN = d.N;
}

int build_descs(mrgan_handle* h) {
  const mrgan_config& c = h->cfg;
  const int B = c.batch, R = h->R, K = c.n_classes, nd = c.noise_dim, nf = h->nf;
  const bool gan = c.model == MRGAN_MODEL_GAN;
  h->h_descs.assign((size_t)NUM_OPS_ALL * nf, GemmDesc{});
  h->h_folds.assign(nf, FoldState{});
  std::vector<BnDesc> bn(nf); std::vector<LossDesc> ls(nf); std::vector<EvalDesc> ev(nf), evs(nf);
  std::vector<AdamRange> rg0(nf), rg1(nf);
  auto setop = [&](int op, int f, GemmDesc d, bool at, bool bt, int rnd = 0) { set_op(h, op, f, d, at, bt, rnd); };
  for (int f = 0; f < nf; ++f) {
    FoldBuffers& b = h->fb[f];
    const int D = h->shapes[f].D;
    const NetLayout& LD = h->net[0][f];
    float* PD = h->P + LD.off; float* GD = h->Gr + LD.off;
    int win[6] = {D, kDW[0], kDW[1], kDW[2], kDW[3], kDW[4]};
    int wout[6] = {kDW[0], kDW[1], kDW[2], kDW[3], kDW[4], K};
    const float sig[5] = {c.sigma_in, c.sigma_hidden, c.sigma_hidden, c.sigma_hidden, c.sigma_hidden};
    const int hact = c.hidden_act == MRGAN_ACT_LEAKY_RELU ? ACT_LEAKY : ACT_RELU;      // mr_gan.py:119-127 / wganlpctsemi.py:169
    const bool dropout = c.dropout > 0.0f;
    // ---- discriminator forward (train): layer l (1-based) reads a[l-1], writes h[l] (+ noisy a[l])
    for (int l = 1; l <= 6; ++l) {
      const TensorLayout& W = LD.t[l - 1];
      float* C = (l <= 5) ? b.hb[l] : b.lg;
      const int ldc = (l <= 5) ? b.lda[l] : pitch8(K);
      GemmDesc d = make_desc(b.a[l - 1], b.lda[l - 1], PD + W.off, W.pitch, C, ldc, R, wout[l - 1], win[l - 1] + 1,
                             EPI_FWD, l <= 5 ? hact : ACT_NONE, f);
      if (l <= 4) { d.C2 = b.a[l]; d.ldc2 = b.lda[l]; d.sigma = sig[l]; d.tid = l; d.row0 = 0; }
      setop(OP_D1 + l - 1, f, d, false, false, (l == 5 ? 1 : 0) | 2);
      if (gan && l <= 5) { GemmDesc dg = d; dg.M = 2 * B; setop(OP_D1G + l - 1, f, dg, false, false, (l == 5 ? 1 : 0) | 2); }
      // eval twin: no noise, reads the clean activations
      const float* EA = (l == 1) ? b.xte : b.eh[l - 1];
      float* EC = (l <= 5) ? b.eh[l] : b.elg;
      GemmDesc e = make_desc(EA, b.lda[l - 1], PD + W.off, W.pitch, EC, ldc, h->shapes[f].n_test, wout[l - 1],
                             win[l - 1] + 1, EPI_FWD, l <= 5 ? hact : ACT_NONE, f);
      setop(l == 1 ? OP_E1 : OP_E2 + l - 2, f, e, false, false, l <= 5 ? 1 : 0);
      if (l == 1) { e.A = b.ex_stage; setop(OP_E1S, f, e, false, false, 1); }
      if (gan) { e.M = B * (h->NE / B); setop(OP_S1 + l - 1, f, e, false, false, l <= 5 ? 1 : 0); }   // generated rows (GenWork)
      // dW (+db): grad(Waug_l) = a[l-1]^T @ dZ[l]
      const float* dZ = (l <= 5) ? b.dz[l] : b.dlg;
      const int lddz = (l <= 5) ? b.ldz[l] : pitch8(K);
      GemmDesc w = make_desc(b.a[l - 1], b.lda[l - 1], dZ, lddz, GD + W.off, W.pitch, win[l - 1] + 1, wout[l - 1], R,
                             EPI_STORE, ACT_NONE, f);
      setop(OP_DW1 + l - 1, f, w, true, false);
      // dX: dZ[l-1] = (dZ[l] @ W_l^T) * relu'(h[l-1])
      if (l >= 2) {
        GemmDesc x = make_desc(dZ, lddz, PD + W.off, W.pitch, b.dz[l - 1], b.ldz[l - 1], R, win[l - 1], wout[l - 1],
                               EPI_DX, hact, f);
        // act'(h[l-1]) needs the layer's clean output -- or, when Dropout follows the activation, the dropped output a[l-1],
        // which carries the keep mask and the sign of h at once (dx_rows); tid >= 1 marks "behind a hidden-layer transform"
        x.aux = (dropout && l - 1 <= 4) ? b.a[l - 1] : b.hb[l - 1]; x.ldaux = b.lda[l - 1]; x.tid = (l - 1 <= 4) ? l - 1 : 0;
        setop(OP_DX2 + l - 2, f, x, false, true, 1);
        if (gan && l <= 5) { GemmDesc xg = x; xg.M = B; setop(OP_DX2G + l - 2, f, xg, false, true, 1); }
        // eval twin: the fold's test rows, act' from the clean activation (phase 0 has no Dropout), and dZ[l-1] written over
        // that activation in place -- the epilogue reads h and writes dZ at the same element, and h is no operand of the GEMM
        // (the ones column at index win[l-1] is outside N and stays)
        GemmDesc ex = make_desc(EC, ldc, PD + W.off, W.pitch, b.eh[l - 1], b.lda[l - 1], h->shapes[f].n_test, win[l - 1], wout[l - 1],
                                EPI_DX, hact, f);
        ex.aux = b.eh[l - 1]; ex.ldaux = b.lda[l - 1]; ex.tid = 0;
        setop(OP_EX2 + l - 2, f, ex, false, true, 1);
      }
    }
    // d/dx = dZ[1] @ W1^T in fp32 (no activation: x is the input), over the staging rows
    const TensorLayout& EW1 = LD.t[0];
    setop(OP_EX1, f, make_desc(b.eh[1], b.lda[1], PD + EW1.off, EW1.pitch, b.ex_stage, b.lda[0], h->shapes[f].n_test, D, kDW[0], EPI_DX,
                               ACT_NONE, f), false, true);
    rg0[f] = AdamRange{LD.off, LD.n};
    ls[f] = LossDesc{b.lg, b.dlg, pitch8(K), b.labels_cur, b.hb[5], b.dz[5], b.lda[5], b.ldz[5], kDW[4]};
    ev[f] = EvalDesc{b.elg, pitch8(K), b.yte, h->shapes[f].n_test, (h->shapes[f].n_test / B) * B, b.eval_out, b.pred};
    evs[f] = EvalDesc{b.elg, pitch8(K), b.ey_stage, h->shapes[f].n_test, 0, b.eval_out_s, b.pred_s};
    if (gan) {
      const NetLayout& LG = h->net[1][f];
      float* PG = h->P + LG.off; float* GG = h->Gr + LG.off;
      const TensorLayout &W1 = LG.t[0], &Tg = LG.t[1], &Tb = LG.t[2], &W2 = LG.t[3], &W3 = LG.t[4];
      const int ldzb = pitch8(nd + 1), ldu = pitch8(kGH + 1), ldx = pitch8(D), ldg = pitch8(kGH);
      setop(OP_G1, f, make_desc(b.zb, ldzb, PG + W1.off, W1.pitch, b.h1g, ldg, B, kGH, nd + 1, EPI_FWD, ACT_SOFTPLUS, f), false, false);
      setop(OP_G2, f, make_desc(b.u, ldu, PG + W2.off, W2.pitch, b.h2g, ldu, B, kGH, kGH + 1, EPI_FWD, ACT_SOFTPLUS, f), false, false, 1);
      GemmDesc g3 = make_desc(b.h2g, ldu, PG + W3.off, W3.pitch, nullptr, 0, B, D, kGH + 1, EPI_FWD, ACT_NONE, f);
      g3.C2 = b.a[0] + (size_t)2 * B * b.lda[0]; g3.ldc2 = b.lda[0]; g3.sigma = c.sigma_in; g3.tid = 0; g3.row0 = 2 * B;
      setop(OP_G3D, f, g3, false, false, 2);
      g3.C2 = b.a[0]; g3.row0 = 0;
      setop(OP_G3G, f, g3, false, false, 2);
      // dFake = dZ[1] @ W1^T  (no activation derivative: fake is G's linear output)
      const TensorLayout& DW1 = LD.t[0];
      setop(OP_DX1G, f, make_desc(b.dz[1], b.ldz[1], PD + DW1.off, DW1.pitch, b.dfake, ldx, B, D, kDW[0], EPI_DX, ACT_NONE, f), false, true, 1);
      setop(OP_GW3, f, make_desc(b.h2g, ldu, b.dfake, ldx, GG + W3.off, W3.pitch, kGH + 1, D, B, EPI_STORE, ACT_NONE, f), true, false);
      GemmDesc gx3 = make_desc(b.dfake, ldx, PG + W3.off, W3.pitch, b.dz2g, ldg, B, kGH, D, EPI_DX, ACT_SOFTPLUS, f);
      gx3.aux = b.h2g; gx3.ldaux = ldu;
      setop(OP_GX3, f, gx3, false, true, 1);
      setop(OP_GW2, f, make_desc(b.u, ldu, b.dz2g, ldg, GG + W2.off, W2.pitch, kGH + 1, kGH, B, EPI_STORE, ACT_NONE, f), true, false);
      setop(OP_GX2, f, make_desc(b.dz2g, ldg, PG + W2.off, W2.pitch, b.du, ldg, B, kGH, kGH, EPI_DX, ACT_NONE, f), false, true);
      setop(OP_GW1, f, make_desc(b.zb, ldzb, b.dz1g, ldg, GG + W1.off, W1.pitch, nd + 1, kGH, B, EPI_STORE, ACT_NONE, f), true, false);
      bn[f] = BnDesc{b.h1g, b.xhat, b.u, b.istd, PG + Tg.off, PG + Tb.off, b.du, b.dz1g, GG + Tg.off, GG + Tb.off,
                     ldg, ldu, B, kGH};
      rg1[f] = AdamRange{LG.off, LG.n};
    }
    FoldState& fs = h->h_folds[f];
    fs.key0 = (uint32_t)(h->shapes[f].seed & 0xFFFFFFFFull);
    fs.key1 = (uint32_t)(h->shapes[f].seed >> 32);
    fs.D = D; fs.n_train = h->shapes[f].n_train; fs.n_test = h->shapes[f].n_test; fs.ldx = pitch8(D);
    fs.x_train = b.xtr; fs.y_train = b.ytr; fs.y_test = b.yte;
    for (int s = 0; s < 3; ++s) fs.idx[s] = b.idx + (size_t)s * h->shapes[f].n_train;
    fs.stage_x = b.stage_x; fs.stage_y = b.stage_y; fs.stage_z = gan ? b.stage_z : nullptr;
    fs.a0 = b.a[0]; fs.lda0 = b.lda[0]; fs.z = gan ? b.zb : nullptr; fs.ldz = pitch8(nd + 1);
    fs.labels_cur = b.labels_cur;
  }
  CK(cudaMemcpy(h->d_descs, h->h_descs.data(), (size_t)NUM_OPS * nf * sizeof(GemmDesc), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_folds, h->h_folds.data(), nf * sizeof(FoldState), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_loss, ls.data(), nf * sizeof(LossDesc), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_eval, ev.data(), nf * sizeof(EvalDesc), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_eval_s, evs.data(), nf * sizeof(EvalDesc), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_ranges[0], rg0.data(), nf * sizeof(AdamRange), cudaMemcpyHostToDevice));
  if (gan) {
    CK(cudaMemcpy(h->d_bn, bn.data(), nf * sizeof(BnDesc), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_ranges[1], rg1.data(), nf * sizeof(AdamRange), cudaMemcpyHostToDevice));
  }
  return MRGAN_OK;
}

// ------------------------------------------------------------------ kernel launch (a failure is kept as the handle's sticky error)
// Every kernel of the library is launched here, so h->launches counts them all.
template <typename... KArgs, typename... Args>
void launch_k(mrgan_handle* h, void (*kern)(KArgs...), const cudaLaunchConfig_t& cfg, Args... args) {
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
  if (e != cudaSuccess && !h->sticky) { h->sticky = MRGAN_ERR_CUDA; h->err = std::string("kernel launch: ") + cudaGetErrorString(e); }
  h->launches++;
}
template <typename... KArgs, typename... Args>
void launch_k(mrgan_handle* h, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  launch_k(h, kern, cfg, args...);
}

void set_ones(mrgan_handle* h, float* p, int ld, int rows, int col) {
  launch_k(h, k_set_col, (rows + 127) / 128, 128, 0, h->stream, p, ld, rows, col, 1.0f, h->om);
}

void init_ones(mrgan_handle* h) {
  const mrgan_config& c = h->cfg;
  const bool gan = c.model == MRGAN_MODEL_GAN;
  for (int f = 0; f < h->nf; ++f) {
    FoldBuffers& b = h->fb[f];
    const int D = h->shapes[f].D;
    int win[6] = {D, kDW[0], kDW[1], kDW[2], kDW[3], kDW[4]};
    set_ones(h, b.a[0], b.lda[0], h->R, D);
    set_ones(h, b.ex_stage, b.lda[0], h->NE, D);
    set_ones(h, b.xte, b.lda[0], h->shapes[f].n_test, D);
    for (int l = 1; l <= 5; ++l) {
      set_ones(h, b.hb[l], b.lda[l], h->R, win[l]);
      if (l < 5) set_ones(h, b.a[l], b.lda[l], h->R, win[l]);
      set_ones(h, b.eh[l], b.lda[l], h->NE, win[l]);
    }
    if (gan) {
      set_ones(h, b.zb, pitch8(c.noise_dim + 1), c.batch, c.noise_dim);
      set_ones(h, b.u, pitch8(kGH + 1), c.batch, kGH);
      set_ones(h, b.h2g, pitch8(kGH + 1), c.batch, kGH);
    }
  }
}


// status of everything enqueued since the last check (launch_k / dp_allreduce record the first failure)
int take_sticky(mrgan_handle* h) {
  if (!h->sticky) return MRGAN_OK;
  const int code = h->sticky;
  h->sticky = 0;
  g_last_error = h->err;
  return code;
}

// ------------------------------------------------------------------ NCCL (resolved at run time: no link dependency)
struct NcclId { char b[128]; };
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;

bool nccl_load() {
  if (g_nccl.lib) return true;
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) return false;
  g_nccl.GetUniqueId = (int (*)(NcclId*))dlsym(lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(lib, "ncclCommInitRank");
  g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(lib, "ncclAllReduce");
  g_nccl.CommDestroy = (int (*)(void*))dlsym(lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy) return false;
  g_nccl.lib = lib;
  return true;
}

// Virtual-rank stand-in for the collective: `buf` holds W equal segments (one per fold = rank); every segment becomes the
// element-wise sum over the segments, added in rank order (what ncclAllReduce(sum) leaves on every rank).
__global__ void k_virtual_allreduce(float* __restrict__ buf, size_t seg, int W) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < seg; i += (size_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < W; ++w) s += buf[(size_t)w * seg + i];
    for (int w = 0; w < W; ++w) buf[(size_t)w * seg + i] = s;
  }
}

// in-stream sum all-reduce of fp32 (ncclFloat32 = 7, ncclSum = 0); no-op outside the data-parallel mode
void dp_allreduce(mrgan_handle* h, float* buf, size_t n) {
  if (h->dp_world <= 1 || n == 0) return;
  if (h->dp_virtual) {
    const size_t seg = n / (size_t)h->dp_world;
    const int blocks = (int)std::min<size_t>((seg + 255) / 256, 1184);
    launch_k(h, k_virtual_allreduce, blocks, 256, 0, h->stream, buf, seg, h->dp_world);
    return;
  }
  const int rc = g_nccl.AllReduce(buf, buf, n, 7, 0, h->nccl_comm, h->stream);
  if (rc != 0 && !h->sticky) {
    h->sticky = MRGAN_ERR_CUDA;
    h->err = std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error");
  }
}

void dp_allreduce_grads(mrgan_handle* h, int net) {
  if (h->dp_world <= 1) return;
  long long n = 0;
  for (int f = 0; f < h->nf; ++f) n += h->net[net][f].n;
  dp_allreduce(h, h->Gr + h->net[net][0].off, (size_t)n);      // the nets of all folds are contiguous in the flat buffer
}

void launch_adam(mrgan_handle* h, int f0, int nfl, int net);

// Pointer sets of the fused exchange.  Real ranks: the same offsets inside every rank's (IPC-mapped) arena.  Virtual ranks:
// fold r's net inside this handle's own flat buffers.
void dp_build_peers(mrgan_handle* h) {
  const float* abase = reinterpret_cast<const float*>(h->arena);
  for (int net = 0; net < 2; ++net) {
    DpPeers& pp = h->dp_peers[net];
    memset(&pp, 0, sizeof(pp));
    if (h->net[net].empty()) continue;
    for (int p = 0; p < h->dp_world; ++p) {
      if (h->dp_virtual) {
        const long long d = h->net[net][p].off - h->net[net][0].off;
        pp.P[p] = h->P + d; pp.Gr[p] = h->Gr + d; pp.Mo[p] = h->Mo + d; pp.Vo[p] = h->Vo + d;
        pp.Ph[p] = h->harena ? h->harena + (h->P - abase) + d : nullptr;
        pp.flags[p] = h->d_dpflags + (size_t)p * DP_FLAG_WORDS;
      } else {
        float* pb = reinterpret_cast<float*>(h->peer_arena[p]);
        pp.P[p] = pb + (h->P - abase); pp.Gr[p] = pb + (h->Gr - abase); pp.Mo[p] = pb + (h->Mo - abase); pp.Vo[p] = pb + (h->Vo - abase);
        pp.Ph[p] = h->peer_harena[p] ? h->peer_harena[p] + (h->P - abase) : nullptr;
        pp.flags[p] = reinterpret_cast<unsigned*>(h->peer_arena[p] + (reinterpret_cast<char*>(h->d_dpflags) - h->arena));
      }
    }
  }
}

// One kernel per rank: reduce-scatter of the net's flat gradient by peer loads, Adam on the owned shard, all-gather of the
// updated weights by peer stores, step counters (kernels_dp.cuh).  Replaces ncclAllReduce + the full-size k_adam.
void dp_exchange(mrgan_handle* h, int net) {
  long long len = 0;
  if (h->dp_virtual) len = h->net[net][0].n;
  else for (int f = 0; f < h->nf; ++f) len += h->net[net][f].n;
  const long long off = h->net[net][0].off;
  const int W = h->dp_world;
  const int bx = h->dp_virtual ? std::max(1, 296 / W) : 296;      // all CTAs co-resident (2 per SM): they wait on one another
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(bx, h->dp_virtual ? W : 1, 1); cfg.blockDim = dim3(256); cfg.stream = h->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const float ginv = h->om.mode == 2 ? 1.0f / h->om.gscale : 1.0f;
  launch_k(h, k_dp_exchange, cfg, h->dp_peers[net], W, h->dp_virtual ? -1 : h->dp_rank, off, len, h->d_folds, h->nf, net, h->hp, ginv);
}

// gradient exchange + optimizer of one net in the data-parallel mode
void dp_update(mrgan_handle* h, int f0, int nfl, int net) {
  if (h->dp_fused) { dp_exchange(h, net); return; }
  dp_allreduce_grads(h, net);
  launch_adam(h, f0, nfl, net);
}

// Scratch of the split (statistics -> [all-reduce] -> apply) BatchNorm / feature-matching kernels: used by the data-parallel
// mode and, on one GPU, by the large-batch regime where one CTA per fold would serialise thousands of rows.
int alloc_split_bufs(mrgan_handle* h) {
  if (h->d_dpbufs) return MRGAN_OK;
  const int nf = h->nf;
  // per fold: the three statistics blocks, the row-chunk partials of the statistics kernels, the block partials of
  // k_loss_disc, and the arrival counters (16 column blocks + 1 for the loss kernel, as 32 words)
  const size_t stats = 2 * kGH + 2 * kGH + 2 * kDW[4];
  const size_t per = stats + (size_t)SPLIT_MAX_Y * 2 * SPLIT_PART_W + 4 * LOSS_MAX_BLOCKS + 32;
  CK(cudaMalloc(&h->d_dpmem, per * nf * sizeof(float)));
  CK(cudaMemset(h->d_dpmem, 0, per * nf * sizeof(float)));
  h->dp_bnf = h->d_dpmem; h->dp_bnb = h->dp_bnf + (size_t)nf * 2 * kGH; h->dp_fm = h->dp_bnb + (size_t)nf * 2 * kGH;
  float* const part = h->dp_fm + (size_t)nf * 2 * kDW[4];
  h->dp_losspart = part + (size_t)nf * SPLIT_MAX_Y * 2 * SPLIT_PART_W;
  unsigned* const ctr = reinterpret_cast<unsigned*>(h->dp_losspart + (size_t)nf * 4 * LOSS_MAX_BLOCKS);
  h->dp_lossctr = ctr + (size_t)nf * 16;
  std::vector<DpBufs> bufs(nf);
  for (int f = 0; f < nf; ++f)
    bufs[f] = DpBufs{h->dp_bnf + (size_t)f * 2 * kGH, h->dp_bnb + (size_t)f * 2 * kGH, h->dp_fm + (size_t)f * 2 * kDW[4],
                     part + (size_t)f * SPLIT_MAX_Y * 2 * SPLIT_PART_W, ctr + (size_t)f * 16};
  CK(cudaMalloc(&h->d_dpbufs, nf * sizeof(DpBufs)));
  CK(cudaMemcpy(h->d_dpbufs, bufs.data(), nf * sizeof(DpBufs), cudaMemcpyHostToDevice));
  return MRGAN_OK;
}

// Row chunks (grid.y) of the split statistics / apply kernels: one chunk per 256 rows (8 rows per thread of a 1024-thread
// block), so that a large batch spreads over the chip instead of 8 - 16 CTAs.
int split_chunks(int rows) {
  const int y = (rows + 255) / 256;
  return y < 1 ? 1 : (y > SPLIT_MAX_Y ? SPLIT_MAX_Y : y);
}

// ------------------------------------------------------------------ launch sequences
// the device descriptors [nf] of op: in the arena's table, or in the workspace of its entry points
const GemmDesc* op_descs(const mrgan_handle* h, int op) {
  if (op < NUM_OPS) return h->d_descs + (size_t)op * h->nf;
  if (op < OP_GG1) return h->sal.descs + (size_t)(op - NUM_OPS) * h->nf;
  return h->gen.descs + (size_t)(op - OP_GG1) * h->nf;
}

// om: where the epilogue's operand copies go (null: the arena's, h->om)
void launch_gemm(mrgan_handle* h, int op, int f0, int nfl, int rows_override, cudaStream_t st = nullptr, const OperandMode* om = nullptr) {
  if (!st) st = h->stream;
  if (h->cfg.precision != MRGAN_PREC_FP32) { tc_launch_gemm(h, op, f0, nfl, rows_override, st, om ? *om : h->om); return; }
  const OpInfo& oi = h->ops[op];
  int M = oi.maxM;
  if (rows_override > 0 && !oi.at) M = rows_override;
  const GemmDesc* d = op_descs(h, op) + f0;
  dim3 grid((oi.maxN + 63) / 64, (M + 63) / 64, nfl);
  if (!oi.at && !oi.bt) launch_k(h, k_gemm_simt<false, false>, grid, dim3(256), 0, st, d, (const FoldState*)h->d_folds, rows_override, h->hp);
  else if (!oi.at && oi.bt) launch_k(h, k_gemm_simt<false, true>, grid, dim3(256), 0, st, d, (const FoldState*)h->d_folds, rows_override, h->hp);
  else launch_k(h, k_gemm_simt<true, false>, grid, dim3(256), 0, st, d, (const FoldState*)h->d_folds, rows_override, h->hp);
}

// side stream: fork = "side waits for everything enqueued on main so far", join = the reverse.
// Works both eagerly and under stream capture (where it becomes graph edges).
void fork_side(mrgan_handle* h) {
  cudaEvent_t e = h->ev_pool[h->ev_next++ & 15];
  cudaEventRecord(e, h->stream);
  cudaStreamWaitEvent(h->side, e, 0);
  h->side_open = true;
}
void join_side(mrgan_handle* h) {
  if (!h->side_open) return;
  h->side_open = false;
  cudaEvent_t e = h->ev_pool[h->ev_next++ & 15];
  cudaEventRecord(e, h->side);
  cudaStreamWaitEvent(h->stream, e, 0);
}

int max_D(const mrgan_handle* h, int f0, int nfl) {
  int m = 0;
  for (int f = f0; f < f0 + nfl; ++f) m = h->shapes[f].D > m ? h->shapes[f].D : m;
  return m;
}

void launch_prep(mrgan_handle* h, int f0, int nfl, int mode, int from_stage, int t, int nrows) {
  const mrgan_config& c = h->cfg;
  int cols = max_D(h, f0, nfl);
  if (c.noise_dim > cols) cols = c.noise_dim;
  // rows per thread: 8 at the reference batch, 16 in the large-batch regime (kernels_simt.cuh: k_prep; 8 / 16 / 32 rows per
  // thread measured the same once the gathers were batched: 224 / 227 / 227 step pairs/s at D = 12032, B = 8192)
  const int pg = nrows > 512 ? 4 : 2;
  dim3 grid((cols + 127) / 128, (nrows + 4 * pg - 1) / (4 * pg), nfl);
#define LAUNCH_PREP(PG) launch_k(h, k_prep<PG>, grid, dim3(128), 0, h->stream, h->d_folds, f0, mode, from_stage, t, c.batch, nrows, c.noise_dim, \
                                 c.sigma_in, h->hp, h->om)
  if (pg == 4) LAUNCH_PREP(4); else LAUNCH_PREP(2);
#undef LAUNCH_PREP
}

void launch_adam(mrgan_handle* h, int f0, int nfl, int net) {
  long long nmax = 0;
  for (int f = f0; f < f0 + nfl; ++f) nmax = h->net[net][f].n > nmax ? h->net[net][f].n : nmax;
  int blocks = (int)((nmax / 4 + 255) / 256);
  if (blocks > 2048) blocks = 2048;
  if (blocks < 1) blocks = 1;
  const AdamRange* ranges = h->d_ranges[net];
  if (h->tc_fused_adam) { ranges = h->d_ranges_tc[net]; blocks = 1; }
  // f16 mode: the gradient buffer carries the loss scale, and every parameter update refreshes the fp16 operand copy
  const float ginv = h->om.mode == 2 ? 1.0f / h->om.gscale : 1.0f;
  __half* Ph = h->om.mode == 2 ? h->harena + (h->P - reinterpret_cast<float*>(h->arena)) : nullptr;
  launch_k(h, k_adam, dim3(blocks, nfl), dim3(256), 0, h->stream, h->P, h->Mo, h->Vo, (const float*)h->Gr, ranges, h->d_folds, f0, net, h->hp,
           ginv, Ph);
}

void enqueue_gen_fwd(mrgan_handle* h, int f0, int nfl, int op_g3) {
  launch_gemm(h, OP_G1, f0, nfl, 0);
  if (h->tc_heads & 4) {                     // BatchNorm ran in G1's epilogue
    launch_gemm(h, OP_G2, f0, nfl, 0);
    launch_gemm(h, op_g3, f0, nfl, 0);
    return;
  }
  const dim3 bnf((kGH + BN_COLS - 1) / BN_COLS, h->d_dpbufs ? split_chunks(h->cfg.batch) : 1, nfl);
  const dim3 bnt(h->cfg.batch > 256 ? 1024 : 256);     // 32 columns x 8 (reference batch) or 32 (large batch) row slices
  const OperandMode tf32 = h->om;
  if (h->d_dpbufs) {          // batch statistics over the GLOBAL batch: local sums -> NVLink all-reduce -> apply
    launch_k(h, k_bn_stats, bnf, bnt, 0, h->stream, h->d_bn + f0, h->d_dpbufs + f0);
    dp_allreduce(h, h->dp_bnf + (size_t)f0 * 2 * kGH, (size_t)nfl * 2 * kGH);
    launch_k(h, k_bn_apply, bnf, bnt, 0, h->stream, h->d_bn + f0, h->d_dpbufs + f0, h->cfg.bn_eps, tf32, h->hp.dp_bg);
  } else {
    launch_k(h, k_bn_fwd, bnf, bnt, 0, h->stream, (const BnDesc*)(h->d_bn + f0), h->cfg.bn_eps, tf32);
  }
  launch_gemm(h, OP_G2, f0, nfl, 0);
  launch_gemm(h, op_g3, f0, nfl, 0);
}

// train_batch_disc (mr_gan.py:169)
void enqueue_disc_step(mrgan_handle* h, int f0, int nfl, int t, int from_stage) {
  const mrgan_config& c = h->cfg;
  const int B = c.batch;
  const bool heads = (h->tc_heads & 1) != 0;
  h->hp.t = t;
  launch_prep(h, f0, nfl, 0, from_stage, t, 2 * B);
  enqueue_gen_fwd(h, f0, nfl, OP_G3D);
  for (int l = 0; l < 6; ++l) launch_gemm(h, OP_D1 + l, f0, nfl, 0);
  if (!heads) {      // otherwise the logit layer's epilogue computed the losses, their gradients and advanced the counters
    // large batch: the 3B rows spread over up to 64 blocks (needs the split scratch for the ordered partial sums)
    int lb = h->dp_losspart ? (3 * B + 511) / 512 : 1;
    lb = lb < 1 ? 1 : (lb > LOSS_MAX_BLOCKS ? LOSS_MAX_BLOCKS : lb);
    launch_k(h, k_loss_disc, dim3(lb, 1, nfl), dim3(256), 0, h->stream, (const LossDesc*)(h->d_loss + f0), h->d_step_stats, f0, h->nf, t, B,
             c.n_classes, c.unlabeled_weight, h->om, h->hp.dp_bg, h->dp_losspart, h->dp_lossctr);
  }
  const bool merge = h->tc_plan[OP_DW3].fused;    // fused dW+Adam: narrow layers may share launches
  for (int l = 6; l >= 1; --l) {      // dX first: it reads W_l, which the fused-Adam dW epilogue overwrites
    if (l >= 2) launch_gemm(h, OP_DX2 + l - 2, f0, nfl, 0);
    if (merge && l > 3) continue;     // the narrow layers 3..6 share ONE dW+Adam launch, after the last dX that reads their weights
    fork_side(h);                     // dW_l (+Adam) streams HBM on the side while main continues the dX chain
    if (merge && l == 3) { tc_launch_dw_adam(h, OP_DW3, 4, f0, nfl, h->side); continue; }
    launch_gemm(h, OP_DW1 + l - 1, f0, nfl, 0, h->side);
  }
  // The side stream's dW kernels read the step's activation buffers (a[l], dZ[l]), which the NEXT step's batch assembly
  // and forward pass overwrite: every step joins the side stream before it ends (measured: deferring the join past the
  // next step's generator forward gains nothing once several fold chains run concurrently, and would need
  // double-buffered activations).
  join_side(h);
  if (h->dp_world > 1) dp_update(h, f0, nfl, 0);
  else if (!heads) launch_adam(h, f0, nfl, 0);
  if (from_stage) dp_allreduce(h, h->d_step_stats + ((size_t)t * h->nf + f0) * 4, (size_t)nfl * 4);
}

// train_batch_gen (mr_gan.py:170)
void enqueue_gen_step(mrgan_handle* h, int f0, int nfl, int t, int from_stage) {
  const mrgan_config& c = h->cfg;
  const int B = c.batch;
  const int hm = h->tc_heads;
  h->hp.t = t;
  launch_prep(h, f0, nfl, 1, from_stage, t, 2 * B);
  enqueue_gen_fwd(h, f0, nfl, OP_G3G);
  for (int l = 0; l < 5; ++l) launch_gemm(h, OP_D1G + l, f0, nfl, 0);
  if (h->d_dpbufs) {
    const dim3 fmg((kDW[4] + BN_COLS - 1) / BN_COLS, split_chunks(B), nfl), fmt(B > 256 ? 1024 : 256);
    launch_k(h, k_fm_stats, fmg, fmt, 0, h->stream, h->d_loss + f0, h->d_dpbufs + f0, B);
    dp_allreduce(h, h->dp_fm + (size_t)f0 * 2 * kDW[4], (size_t)nfl * 2 * kDW[4]);
    launch_k(h, k_fm_apply, fmg, fmt, 0, h->stream, h->d_loss + f0, h->d_dpbufs + f0, h->d_step_stats, f0, h->nf, t, B,
             h->om, h->hp.dp_bg, h->dp_world, h->hp.alpha);
  } else if (!(hm & 2)) {   // otherwise D layer 5's epilogue computed the feature-matching loss, its gradient, and advanced the counters
    launch_k(h, k_fm, dim3(1, 1, nfl), dim3(1024), 0, h->stream, (const LossDesc*)(h->d_loss + f0), h->d_step_stats, f0, h->nf, t, B,
             h->om, h->hp.alpha);
  }
  for (int l = 5; l >= 2; --l) launch_gemm(h, OP_DX2G + l - 2, f0, nfl, 0);
  launch_gemm(h, OP_DX1G, f0, nfl, 0);
  launch_gemm(h, OP_GX3, f0, nfl, 0);
  fork_side(h);
  launch_gemm(h, OP_GW3, f0, nfl, 0, h->side);
  launch_gemm(h, OP_GX2, f0, nfl, 0);
  const bool merge = h->tc_plan[OP_GW1].fused;
  if (!merge) {
    fork_side(h);
    launch_gemm(h, OP_GW2, f0, nfl, 0, h->side);
  }
  const dim3 bng((kGH + BN_COLS - 1) / BN_COLS, h->d_dpbufs ? split_chunks(B) : 1, nfl), bnt(B > 256 ? 1024 : 256);
  if (h->d_dpbufs) {
    launch_k(h, k_bn_bwd_stats, bng, bnt, 0, h->stream, h->d_bn + f0, h->d_dpbufs + f0, h->om);
    dp_allreduce(h, h->dp_bnb + (size_t)f0 * 2 * kGH, (size_t)nfl * 2 * kGH);
    launch_k(h, k_bn_bwd_apply, bng, bnt, 0, h->stream, h->d_bn + f0, h->d_dpbufs + f0, h->om, h->hp.dp_bg);
  } else {
    launch_k(h, k_bn_bwd, bng, bnt, 0, h->stream, (const BnDesc*)(h->d_bn + f0), h->om);
  }
  fork_side(h);
  if (merge) tc_launch_dw_adam(h, OP_GW1, 2, f0, nfl, h->side);      // G layers 1 and 2 share one dW+Adam launch
  else launch_gemm(h, OP_GW1, f0, nfl, 0, h->side);
  join_side(h);
  if (h->dp_world > 1) dp_update(h, f0, nfl, 1);
  else launch_adam(h, f0, nfl, 1);      // gamma / beta and the generator's step counters
  dp_allreduce(h, h->d_step_stats + ((size_t)t * h->nf + f0) * 4, (size_t)nfl * 4);
}

// one model.fit batch of mr_nn (mr_nn.py:117)
void enqueue_nn_step(mrgan_handle* h, int f0, int nfl, int t, int from_stage, int n) {
  const mrgan_config& c = h->cfg;
  // a ragged batch (n < batch) runs at full height: k_loss_mse zeroes the gradient rows >= n, so the
  // stale rows contribute nothing to dW/db and every GEMM keeps its static shape
  h->hp.t = t;
  launch_prep(h, f0, nfl, 2, from_stage, t, n);
  for (int l = 0; l < 6; ++l) launch_gemm(h, OP_D1 + l, f0, nfl, 0);
  launch_k(h, k_loss_mse, dim3(1, 1, nfl), dim3(256), 0, h->stream, (const LossDesc*)(h->d_loss + f0), h->d_step_stats, f0, h->nf, t, n, h->R,
           c.n_classes, h->om);
  for (int l = 6; l >= 1; --l) {
    if (l >= 2) launch_gemm(h, OP_DX2 + l - 2, f0, nfl, 0);
    fork_side(h);
    launch_gemm(h, OP_DW1 + l - 1, f0, nfl, 0, h->side);
  }
  join_side(h);
  launch_adam(h, f0, nfl, 0);
}

// test_batch (mr_gan.py:171): phase 0, no noise; with_pred: also the predicted class of every row (fb[f].pred / pred_s)
void enqueue_eval(mrgan_handle* h, int f0, int nfl, bool staged, int n_override, bool with_pred = false) {
  join_side(h);
  launch_gemm(h, staged ? OP_E1S : OP_E1, f0, nfl, n_override);
  for (int l = 1; l < 6; ++l) launch_gemm(h, OP_E2 + l - 1, f0, nfl, n_override);
  launch_k(h, k_argmax_err, dim3(1, 1, nfl), dim3(256), 0, h->stream, (const EvalDesc*)((staged ? h->d_eval_s : h->d_eval) + f0), n_override,
           h->cfg.n_classes, (int)with_pred);
}

// confusion counts of folds [0, nf) from the EvalDesc rows (y, pred) -> h->d_conf
void enqueue_confusion(mrgan_handle* h) {
  const int K = h->cfg.n_classes;
  int nmax = 1;
  for (int f = 0; f < h->nf; ++f) nmax = std::max(nmax, h->shapes[f].n_test);
  cudaMemsetAsync(h->d_conf, 0, (size_t)h->nf * K * K * sizeof(int), h->stream);
  launch_k(h, k_confusion, dim3((nmax + CONF_ROWS - 1) / CONF_ROWS, h->nf), dim3(256), 0, h->stream, (const EvalDesc*)h->d_eval, K, h->d_conf);
}

// Input gradients d log softmax(l)_t / dx of the phase-0 logits l of folds [f0, f0 + nfl) (mrgan_input_grad / mrgan_saliency):
// the eval forward, the seed e_t - softmax(l) over the logits, then the dX chain OP_EX6 .. OP_EX2 over the eval activations (each
// dZ over the activation it came from) and OP_EX1 into ex_stage, fp32.  Targets: the rows' predicted classes (TGT_PRED), the
// resident test labels (TGT_TEST) or the staged labels (TGT_STAGED).  Needs saliency_setup.
enum { TGT_PRED = 0, TGT_TEST = 1, TGT_STAGED = 2 };
void enqueue_input_grad(mrgan_handle* h, int f0, int nfl, bool staged, int n_override, int tgt) {
  enqueue_eval(h, f0, nfl, staged, n_override);
  int n = n_override;
  for (int f = f0; f < f0 + nfl && n_override <= 0; ++f) n = std::max(n, h->shapes[f].n_test);
  launch_k(h, k_logprob_seed, dim3((n + 255) / 256, 1, nfl), dim3(256), 0, h->stream,
           (const EvalDesc*)((tgt == TGT_STAGED ? h->d_eval_s : h->d_eval) + f0), n_override, h->cfg.n_classes, (int)(tgt == TGT_PRED), h->om);
  for (int l = 6; l >= 1; --l) launch_gemm(h, l >= 2 ? OP_EX2 + l - 2 : OP_EX1, f0, nfl, n_override);
  if (h->om.mode == 2)
    launch_k(h, k_unscale_grad, dim3(std::min((n * max_D(h, f0, nfl) + 255) / 256, 1184), 1, nfl), dim3(256), 0, h->stream,
             (const GemmDesc*)(h->sal.descs + (size_t)(OP_EX1 - NUM_OPS) * h->nf + f0), n_override, 1.0f / h->om.gscale);
}

// mrgan_saliency's pass over every fold's resident test set: input gradients for the true classes, then the class means
void enqueue_saliency(mrgan_handle* h) {
  const int Dmax = max_D(h, 0, h->nf);
  enqueue_input_grad(h, 0, h->nf, false, 0, TGT_TEST);
  launch_k(h, k_saliency, dim3((Dmax + 127) / 128, h->nf), dim3(128), 0, h->stream,
           (const GemmDesc*)(h->sal.descs + (size_t)(OP_EX1 - NUM_OPS) * h->nf), (const EvalDesc*)h->d_eval, h->cfg.n_classes, Dmax, h->sal.profile);
}

// the workspace of the input-gradient entry points (descriptors of the OP_EX* ops, the profile), on first use
int saliency_setup(mrgan_handle* h) {
  mrgan_handle::SalWork& S = h->sal;
  if (S.mem) return MRGAN_OK;
  const int nf = h->nf;
  const bool tc = h->cfg.precision != MRGAN_PREC_FP32;
  auto layout = [&](Arena& ar) {
    S.descs = ar.take<GemmDesc>((size_t)NUM_EX * nf);
    S.profile = ar.take<float>((size_t)nf * h->cfg.n_classes * max_D(h, 0, nf));
    S.tcops = tc ? ar.take<TcOp>((size_t)NUM_EX * nf) : nullptr;
  };
  Arena sizing;
  layout(sizing);
  char* mem = nullptr;
  CK(cudaMalloc(&mem, sizing.off + 256));
  Arena real; real.base = mem;
  layout(real);
  int rc = MRGAN_OK;
  if (cudaMemcpy(S.descs, h->h_descs.data() + (size_t)NUM_OPS * nf, (size_t)NUM_EX * nf * sizeof(GemmDesc), cudaMemcpyHostToDevice) != cudaSuccess)
    rc = fail(h, MRGAN_ERR_CUDA, "saliency workspace: descriptor upload failed");
  if (rc == MRGAN_OK && tc) rc = tc_views(h, NUM_OPS, OP_GG1, S.tcops);
  if (rc != MRGAN_OK) { cudaFree(mem); return rc; }
  S.mem = mem;
  return MRGAN_OK;
}

void gen_free(mrgan_handle* h) {
  mrgan_handle::GenWork& G = h->gen;
  if (G.mem) cudaFree(G.mem);
  if (G.hmem) cudaFree(G.hmem);
  G = mrgan_handle::GenWork();
}

// The workspace of the sample entry points, on first use: the generator's activations of NG rows per fold, the descriptors of
// OP_GG* (built here: they point into the workspace) and OP_S* (built with the handle), the BatchNorm segments, the statistics
// descriptors and accumulators.  Ones columns: z's is written with every draw (k_gen_z), u's and h2's once here.
int gen_setup(mrgan_handle* h) {
  mrgan_handle::GenWork& G = h->gen;
  if (G.mem) return MRGAN_OK;
  const mrgan_config& c = h->cfg;
  const int nf = h->nf, B = c.batch, nd = c.noise_dim, NG = B * (h->NE / B), NS = NG / B;
  const int ldz = pitch8(nd + 1), ldg = pitch8(kGH), ldu = pitch8(kGH + 1);
  const bool tc = c.precision != MRGAN_PREC_FP32;
  std::vector<float*> u(nf), h2(nf), h1(nf), xh(nf), is(nf), xo(nf);
  size_t hfloats = 0;
  auto layout = [&](Arena& ar) {
    G.z = ar.take<float>((size_t)nf * NG * ldz);          // operands first: the fp16 shadow covers [0, hfloats)
    for (int f = 0; f < nf; ++f) { u[f] = ar.take<float>((size_t)NG * ldu); h2[f] = ar.take<float>((size_t)NG * ldu); }
    hfloats = (ar.off + 255) / 256 * 256 / sizeof(float);
    G.zs = ar.take<float>((size_t)NG * nd);
    for (int f = 0; f < nf; ++f) {
      h1[f] = ar.take<float>((size_t)NG * ldg); xh[f] = ar.take<float>((size_t)NG * ldg);
      is[f] = ar.take<float>((size_t)NS * ldg); xo[f] = ar.take<float>((size_t)NG * pitch8(h->shapes[f].D));
    }
    G.descs = ar.take<GemmDesc>((size_t)NUM_GEN * nf);
    G.tcops = tc ? ar.take<TcOp>((size_t)NUM_GEN * nf) : nullptr;
    G.bn = ar.take<BnDesc>((size_t)nf * NS);
    G.st = ar.take<StatsDesc>((size_t)2 * nf);
    G.s1 = ar.take<double>((size_t)nf * 2 * SS_W);
    G.s2 = ar.take<double>((size_t)nf * 2 * SS_W * SS_W);
    G.score = ar.take<double>((size_t)nf * 2);
    G.counts = ar.take<int>((size_t)nf * 64);
  };
  Arena sizing;
  layout(sizing);
  char* mem = nullptr;
  CK(cudaMalloc(&mem, sizing.off + 256));
  G.mem = mem;                  // from here on gen_free releases everything on a failed return
  Arena real; real.base = mem;
  layout(real);
  G.om = h->om; G.om.fbase = reinterpret_cast<const float*>(mem); G.om.hbase = nullptr;
  G.hfloats = hfloats; G.NG = NG; G.nseg = NS; G.ldz = ldz; G.zstride = (size_t)NG * ldz;
  auto bail = [&](int rc) { gen_free(h); return rc; };
  if (cudaMemset(mem, 0, sizing.off + 256) != cudaSuccess) return bail(fail(h, MRGAN_ERR_CUDA, "sample workspace: cudaMemset failed"));
  if (h->om.mode == 2) {        // pad columns of the copies are zero like those of the fp32 buffers
    if (cudaMalloc(&G.hmem, hfloats * sizeof(__half)) != cudaSuccess || cudaMemset(G.hmem, 0, hfloats * sizeof(__half)) != cudaSuccess)
      return bail(fail(h, MRGAN_ERR_CUDA, "sample workspace: fp16 shadow allocation failed"));
    G.om.hbase = G.hmem;
  }
  std::vector<BnDesc> bn((size_t)nf * NS);
  std::vector<StatsDesc> st((size_t)2 * nf);
  for (int f = 0; f < nf; ++f) {
    const FoldBuffers& b = h->fb[f];
    const NetLayout& LG = h->net[1][f];
    const float* PG = h->P + LG.off;
    const TensorLayout &W1 = LG.t[0], &Tg = LG.t[1], &Tb = LG.t[2], &W2 = LG.t[3], &W3 = LG.t[4];
    const int D = h->shapes[f].D;
    float* z = G.z + (size_t)f * G.zstride;
    set_op(h, OP_GG1, f, make_desc(z, ldz, PG + W1.off, W1.pitch, h1[f], ldg, NG, kGH, nd + 1, EPI_FWD, ACT_SOFTPLUS, f), false, false, 0);
    set_op(h, OP_GG2, f, make_desc(u[f], ldu, PG + W2.off, W2.pitch, h2[f], ldu, NG, kGH, kGH + 1, EPI_FWD, ACT_SOFTPLUS, f), false, false, 1);
    GemmDesc g3 = make_desc(h2[f], ldu, PG + W3.off, W3.pitch, xo[f], pitch8(D), NG, D, kGH + 1, EPI_FWD, ACT_NONE, f);
    g3.C2 = b.ex_stage; g3.ldc2 = b.lda[0];          // sigma = 0: the clean rows again, as D's first operand
    set_op(h, OP_GG3, f, g3, false, false, 2);
    for (int s = 0; s < NS; ++s) {
      const size_t r = (size_t)s * B;
      bn[(size_t)f * NS + s] = BnDesc{h1[f] + r * ldg, xh[f] + r * ldg, u[f] + r * ldu, is[f] + (size_t)s * ldg, PG + Tg.off, PG + Tb.off,
                                      nullptr, nullptr, nullptr, nullptr, ldg, ldu, B, kGH};
    }
    for (int side = 0; side < 2; ++side)
      st[(size_t)side * nf + f] = StatsDesc{b.eh[5], b.elg, b.lda[5], pitch8(c.n_classes), side ? h->shapes[f].n_test : NG,
                                            G.s1 + ((size_t)f * 2 + side) * SS_W, G.s2 + ((size_t)f * 2 + side) * SS_W * SS_W,
                                            G.score + (size_t)f * 2 + side, side ? nullptr : G.counts + (size_t)f * 64};
    launch_k(h, k_set_col, (NG + 127) / 128, 128, 0, h->stream, u[f], ldu, NG, kGH, 1.0f, G.om);
    launch_k(h, k_set_col, (NG + 127) / 128, 128, 0, h->stream, h2[f], ldu, NG, kGH, 1.0f, G.om);
  }
  if (cudaMemcpy(G.descs, h->h_descs.data() + (size_t)OP_GG1 * nf, (size_t)NUM_GEN * nf * sizeof(GemmDesc), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(G.bn, bn.data(), bn.size() * sizeof(BnDesc), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(G.st, st.data(), st.size() * sizeof(StatsDesc), cudaMemcpyHostToDevice) != cudaSuccess)
    return bail(fail(h, MRGAN_ERR_CUDA, "sample workspace: descriptor upload failed"));
  if (tc) { const int rc = tc_views(h, OP_GG1, NUM_OPS_ALL, G.tcops); if (rc != MRGAN_OK) return bail(rc); }
  if (cudaStreamSynchronize(h->stream) != cudaSuccess) return bail(fail(h, MRGAN_ERR_CUDA, "sample workspace: ones columns failed"));
  const int sk = take_sticky(h);
  return sk != MRGAN_OK ? bail(sk) : MRGAN_OK;
}

// G's forward over rows [r0, r0 + c) of a request (c: whole batches, at most NG) for folds [f0, f0 + nfl): z (drawn, or with
// staged the caller's rows in zs, one fold), OP_GG1, BatchNorm with the statistics of each batch of the chunk (mr_gan.py:112
// in training phase: the only way G ever ran), OP_GG2, OP_GG3 -> the clean rows and their operand copy in ex_stage.
void enqueue_generate(mrgan_handle* h, int f0, int nfl, int r0, int c, uint32_t seed, bool staged) {
  const mrgan_handle::GenWork& G = h->gen;
  const int nd = h->cfg.noise_dim, B = h->cfg.batch, ns = c / B;
  launch_k(h, k_gen_z, dim3((nd + 128) / 128, ((r0 + c - 1) >> 2) - (r0 >> 2) + 1, nfl), 128, 0, h->stream, (const FoldState*)h->d_folds, f0,
           G.z + (size_t)f0 * G.zstride, G.zstride, G.ldz, staged ? (const float*)G.zs : nullptr, r0, c, nd, seed, G.om);
  launch_gemm(h, OP_GG1, f0, nfl, c, nullptr, &G.om);
  // one BnDesc per (fold, segment): a chunk of whole segments is one launch; a short chunk of several folds one per fold
  const dim3 bgx((kGH + BN_COLS - 1) / BN_COLS), bnt(B > 256 ? 1024 : 256);
  if (ns == G.nseg || nfl == 1)
    launch_k(h, k_bn_fwd, dim3(bgx.x, 1, nfl * ns), bnt, 0, h->stream, (const BnDesc*)(G.bn + (size_t)f0 * G.nseg), h->cfg.bn_eps, G.om);
  else
    for (int f = f0; f < f0 + nfl; ++f)
      launch_k(h, k_bn_fwd, dim3(bgx.x, 1, ns), bnt, 0, h->stream, (const BnDesc*)(G.bn + (size_t)f * G.nseg), h->cfg.bn_eps, G.om);
  launch_gemm(h, OP_GG2, f0, nfl, c, nullptr, &G.om);
  launch_gemm(h, OP_GG3, f0, nfl, c);
}

// mrgan_sample_stats's pass over every fold: n generated rows in chunks of NG (z from seed), each through D's eval forward
// (OP_S*) and into the accumulators, then the resident test rows (OP_E*).  Needs gen_setup.
void enqueue_sample_stats(mrgan_handle* h, int n, uint32_t seed) {
  const mrgan_handle::GenWork& G = h->gen;
  const int nf = h->nf, K = h->cfg.n_classes;
  cudaMemsetAsync(G.s1, 0, (size_t)(reinterpret_cast<char*>(G.counts + (size_t)nf * 64) - reinterpret_cast<char*>(G.s1)), h->stream);
  for (int r0 = 0; r0 < n; r0 += G.NG) {
    const int c = std::min(G.NG, n - r0);
    enqueue_generate(h, 0, nf, r0, c, seed, false);
    for (int l = 0; l < 6; ++l) launch_gemm(h, OP_S1 + l, 0, nf, c);
    launch_k(h, k_sample_stats, dim3(SS_TILES + 1, nf), SS_THREADS, 0, h->stream, (const StatsDesc*)G.st, c, K);
  }
  for (int l = 0; l < 6; ++l) launch_gemm(h, l == 0 ? OP_E1 : OP_E2 + l - 1, 0, nf, 0);
  launch_k(h, k_sample_stats, dim3(SS_TILES + 1, nf), SS_THREADS, 0, h->stream, (const StatsDesc*)(G.st + nf), 0, K);
}

int finish_pending(mrgan_handle* h) {
  if (h->epoch_pending) {
    CK(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->last_ms = ms;
    h->epoch_pending = false;
  }
  return MRGAN_OK;
}

#define TRY(expr)                                                                                  \
  do {                                                                                             \
    const int _rc = (expr);                                                                        \
    if (_rc) return _rc;                                                                           \
  } while (0)

// What a C-ABI entry point needs of its handle.  Every entry point that takes a handle and returns a status calls
// enter() first and ready() after its own argument checks, so the checks run in one order (enter reads FOLD and the
// model flags, ready reads FOLD and the state flags):
//   enter: null handle, fold index (MRGAN_ERR_ARG); model (MRGAN_ERR_STATE)
//   ... the call's own argument checks (MRGAN_ERR_ARG) ...
//   ready: data-parallel mode, loaded folds, fitted SVM (MRGAN_ERR_STATE); then the handle's device and a pending epoch.
enum : unsigned {
  FOLD = 1u,          // the call takes a fold index
  GAN = 2u, NN = 4u, SVM = 8u,
  NETS = 16u,         // GAN or NN: an SVM handle has no nets
  LOADED = 32u,       // the call's fold, or every fold of the handle, has its data (mrgan_load_fold / mrgan_prepare_fold)
  FITTED = 64u,       // mrgan_svm_fit* ran since the last invalidation
  LOCAL = 128u,       // not a data-parallel handle (mrgan_dp_init / mrgan_dp_init_virtual)
  NOT_VIRTUAL = 256u, // not a handle whose folds play virtual ranks
};

int enter(mrgan_handle* h, const char* fn, unsigned need, int fold = 0) {
  if (!h) return fail(nullptr, MRGAN_ERR_ARG, "null handle");
  if ((need & FOLD) && (fold < 0 || fold >= h->nf)) return fail(h, MRGAN_ERR_ARG, "fold index out of range");
  const int m = h->cfg.model;
  if ((need & GAN) && m != MRGAN_MODEL_GAN) return fail(h, MRGAN_ERR_STATE, std::string(fn) + " needs a GAN handle");
  if ((need & NN) && m != MRGAN_MODEL_NN) return fail(h, MRGAN_ERR_STATE, std::string(fn) + " needs an NN handle");
  if ((need & SVM) && m != MRGAN_MODEL_SVM) return fail(h, MRGAN_ERR_STATE, std::string(fn) + " needs an SVM handle");
  if ((need & NETS) && m == MRGAN_MODEL_SVM) return fail(h, MRGAN_ERR_STATE, std::string(fn) + ": not available on an SVM handle");
  return MRGAN_OK;
}

int ready(mrgan_handle* h, const char* fn, unsigned need, int fold = 0) {
  if ((need & LOCAL) && (h->dp_world > 1 || h->dp_virtual || h->nccl_comm))
    return fail(h, MRGAN_ERR_STATE, std::string(fn) + ": not available on a data-parallel handle");
  if ((need & NOT_VIRTUAL) && h->dp_virtual)
    return fail(h, MRGAN_ERR_STATE, std::string(fn) + ": virtual ranks step together: use mrgan_train_epoch");
  if (need & LOADED)
    for (int f = (need & FOLD) ? fold : 0; f < ((need & FOLD) ? fold + 1 : h->nf); ++f)
      if (!h->fb[f].loaded) return fail(h, MRGAN_ERR_STATE, std::string(fn) + " before mrgan_load_fold");
  if ((need & FITTED) && !h->svm.fitted) return fail(h, MRGAN_ERR_STATE, std::string(fn) + " before mrgan_svm_fit");
  CK(cudaSetDevice(h->cfg.device));
  return finish_pending(h);
}

// The end of an entry point that enqueued work: wait for it, then report a failed launch or collective.
int complete(mrgan_handle* h) {
  CK(cudaStreamSynchronize(h->stream));
  CKS();
  return MRGAN_OK;
}

// Average device ms of `reps` calls of once() on the handle's stream, after one warm-up call.
template <typename Once>
int time_reps(mrgan_handle* h, int reps, Once once, float* ms_avg) {
  once();
  CK(cudaEventRecord(h->ev0, h->stream));
  for (int i = 0; i < reps; ++i) once();
  CK(cudaEventRecord(h->ev1, h->stream));
  TRY(complete(h));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  *ms_avg = ms / reps;
  return MRGAN_OK;
}

// Rows that feed the first eval MMA directly get their operand form: rounded onto the tf32 grid (RN), or their fp16 copy.
void to_operand(mrgan_handle* h, float* p, size_t n) {
  if (h->cfg.precision == MRGAN_PREC_TF32) launch_k(h, k_round_tf32, 256, 256, 0, h->stream, p, n);
  else if (h->om.mode == 2) launch_k(h, k_to_half, 256, 256, 0, h->stream, p, n, h->om);
}

// Host rows x [n][D] of a fold -> its eval staging rows (ex_stage), in operand form.
int stage_rows(mrgan_handle* h, int fold, const float* x, int n) {
  FoldBuffers& b = h->fb[fold];
  const size_t w = (size_t)h->shapes[fold].D * sizeof(float);
  CK(cudaMemcpy2DAsync(b.ex_stage, (size_t)b.lda[0] * sizeof(float), x, w, w, n, cudaMemcpyHostToDevice, h->stream));
  to_operand(h, b.ex_stage, (size_t)n * b.lda[0]);
  return MRGAN_OK;
}

// The captured epochs bake in the handle's mode: a mode change drops them, and the next epoch captures again.
void drop_graphs(mrgan_handle* h) {
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second);
  h->graphs.clear(); h->graph_nodes.clear();
}

// The handle becomes a data-parallel replica of `world` ranks (rank < 0: its folds play the ranks).
int dp_switch(mrgan_handle* h, int world, int rank) {
  TRY(alloc_split_bufs(h));
  h->dp_world = world; h->dp_rank = std::max(rank, 0); h->dp_virtual = rank < 0;
  h->hp.dp_bloc = h->cfg.batch; h->hp.dp_bg = h->cfg.batch * world; h->hp.dp_rank = rank;     // -1: rank = fold index (common.cuh)
  if (h->cfg.precision != MRGAN_PREC_FP32) {   // gradients must be all-reduced before Adam: dW stores them, k_adam applies
    tc_teardown(h);
    h->tc_fused_adam = false;
    TRY(tc_setup(h));
  }
  drop_graphs(h);
  CK(cudaDeviceSynchronize());
  return MRGAN_OK;
}

// Device temporaries of one call, freed on every return path.
struct Temps {
  std::vector<void*> p;
  template <typename T> cudaError_t alloc(T** ptr, size_t bytes) {
    const cudaError_t e = cudaMalloc(ptr, bytes);
    if (e == cudaSuccess) p.push_back(*ptr);
    return e;
  }
  ~Temps() { for (void* q : p) cudaFree(q); }
};

// reference-order <-> internal (augmented, padded) parameter layout
void pack_params(const mrgan_handle* h, int fold, int net, const float* src, std::vector<float>& dst, bool to_internal,
                 float* out_ref) {
  const NetLayout& L = h->net[net][fold];
  long long o = 0;
  auto mat = [&](const TensorLayout& t, int rows_w) {     // W[rows_w, cols] then b[cols]
    for (int r = 0; r < rows_w + 1; ++r)
      for (int cidx = 0; cidx < t.cols; ++cidx) {
        const long long ii = t.off + (long long)r * t.pitch + cidx;
        if (to_internal) dst[ii] = src[o]; else out_ref[o] = dst[ii];
        ++o;
      }
  };
  auto vec = [&](const TensorLayout& t) {
    for (int cidx = 0; cidx < t.cols; ++cidx) {
      if (to_internal) dst[t.off + cidx] = src[o]; else out_ref[o] = dst[t.off + cidx];
      ++o;
    }
  };
  if (net == 0) {
    for (int l = 0; l < 6; ++l) mat(L.t[l], L.t[l].rows - 1);
  } else {
    mat(L.t[0], L.t[0].rows - 1); vec(L.t[1]); vec(L.t[2]); mat(L.t[3], L.t[3].rows - 1); mat(L.t[4], L.t[4].rows - 1);
  }
}

int build_graph(mrgan_handle* h, int key, int nb) {
  if (h->graphs.count(key)) return MRGAN_OK;
  const mrgan_config& c = h->cfg;
  const long long before = h->launches;
  cudaGraph_t g = nullptr;
  CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  {
    cudaStream_t origin = h->stream, origin_side = h->side;
    const int nch = h->dp_world > 1 ? 1 : h->nchains;      // collectives: one chain, the same order on every rank
    cudaEvent_t e = h->ev_pool[h->ev_next++ & 15];
    cudaEventRecord(e, origin);
    for (int ch = 1; ch < nch; ++ch) cudaStreamWaitEvent(h->cmain[ch], e, 0);
    for (int ch = 0; ch < nch; ++ch) {
      const int f0 = (int)((long long)h->nf * ch / nch), f1 = (int)((long long)h->nf * (ch + 1) / nch);
      if (f1 <= f0) continue;
      h->stream = h->cmain[ch]; h->side = h->cside[ch];
      h->side_open = false;
      if (c.model == MRGAN_MODEL_GAN) {
        for (int t = 0; t < nb; ++t) {
          enqueue_disc_step(h, f0, f1 - f0, t, 0);
          enqueue_gen_step(h, f0, f1 - f0, t, 0);
        }
        if (c.eval_each_epoch) enqueue_eval(h, f0, f1 - f0, false, 0);
        join_side(h);                             // every forked stream must rejoin before the capture ends
      } else {
        for (int t = 0; t < nb; ++t) enqueue_nn_step(h, f0, f1 - f0, t, 0, c.batch);
        join_side(h);
      }
    }
    h->stream = origin; h->side = origin_side;
    for (int ch = 1; ch < nch; ++ch) {
      cudaEvent_t j = h->ev_pool[h->ev_next++ & 15];
      cudaEventRecord(j, h->cmain[ch]);
      cudaStreamWaitEvent(origin, j, 0);
    }
  }
  launch_k(h, k_epoch_reduce, h->nf, 32, 0, h->stream, h->d_step_stats, h->d_eval, h->d_epoch_stats, h->nf, nb,
           (int)(c.model == MRGAN_MODEL_GAN && c.eval_each_epoch));
  CK(cudaMemcpyAsync(h->h_epoch_stats, h->d_epoch_stats, (size_t)h->nf * 8 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamEndCapture(h->stream, &g));
  { const int sk = take_sticky(h); if (sk) { cudaGraphDestroy(g); return sk; } }
  cudaGraphExec_t ge = nullptr;
  CK(cudaGraphInstantiate(&ge, g, 0));
  CK(cudaGraphDestroy(g));
  h->graphs[key] = ge;
  h->graph_nodes[key] = h->launches - before;
  h->launches = before;
  return MRGAN_OK;
}

int upload_indices(mrgan_handle* h, const int32_t* const* streams, int n_streams, int n_idx) {
  // host [nf][n_idx] per stream -> pinned staging -> device idx[f][s][n_train]
  const int slot = h->idx_slot;
  h->idx_slot ^= 1;
  CK(cudaEventSynchronize(h->idx_free[slot]));
  int* pin = h->h_idx_pinned[slot];
  for (int f = 0; f < h->nf; ++f)
    for (int s = 0; s < n_streams; ++s)
      memcpy(pin + ((size_t)f * 3 + s) * h->n_train, streams[s] + (size_t)f * n_idx, (size_t)n_idx * sizeof(int));
  for (int f = 0; f < h->nf; ++f)
    CK(cudaMemcpyAsync(h->fb[f].idx, pin + (size_t)f * 3 * h->n_train, (size_t)3 * h->n_train * sizeof(int),
                       cudaMemcpyHostToDevice, h->stream));
  CK(cudaEventRecord(h->idx_free[slot], h->stream));
  return MRGAN_OK;
}

}  // namespace


// ------------------------------------------------------------------ tcgen05 path: host side
namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2D fp32 tensor [rows, cols] with `pitch` floats per row; box = 32 columns (one 128B swizzle row) x box_rows
// L2 promotion of the TMA loads: every box row is one 128-byte line of a row-major matrix, so neighbouring boxes /
// k-blocks touch the adjacent 128 bytes of the same DRAM page; fetching 256 B per miss halves the DRAM activations.
constexpr CUtensorMapL2promotion kL2Promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;

// esz = 4: fp32 elements (read as tf32); esz = 2: fp16 elements (`base` then points at __half data, pitch in elements).
// The swizzled box is always one 128-byte row wide (32 fp32 / 64 fp16 elements); MN-major 32-bit operands need the
// 32-byte-atom variant of the 128B swizzle, 16-bit ones the plain 128B swizzle.
bool make_map(EncodeTiledFn fn, CUtensorMap* m, const void* base, int cols, int rows, int pitch, int box_rows,
              bool mn_major, int box_cols = 0, int esz = 4) {
  const int row_elems = 128 / esz;
  if (box_cols == 0) box_cols = row_elems;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch * (cuuint64_t)esz};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1u, 1u};
  return fn(m, esz == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims,
            strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            box_cols != row_elems ? CU_TENSOR_MAP_SWIZZLE_NONE
                                  : ((mn_major && esz == 4) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B),
            kL2Promo,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

// forward / dX: 4-stage ring, up to 256 accumulator columns, 1 CTA per SM
// dW (+ fused Adam): 2-stage ring (the contraction is only ~150 rows = 5 blocks), 128 columns, 2 CTAs per SM
// large-batch regime (more than 256 batch rows: data-parallel config 5): 256 x 256 tiles, 3-stage ring of 64 KB stages
#define TC_FWD_STAGES 4
#define TC_DW_STAGES 2
#define TC_BIG_STAGES 3
#define TC_FWD_THREADS (64 + 32 * 8)
#define TC_DW_THREADS (64 + 32 * 4)
constexpr int kTcSmemMax = 227 * 1024;     // the most dynamic shared memory a block may have
constexpr size_t tc_smem_bytes(int bn, int stages, int mt = 1) { return 1024 + (size_t)stages * ((size_t)mt * 128 * 128 + (size_t)bn * 128) + 256; }

// The k_gemm_tc instantiations the library launches, by role, operand format F (false: fp32 operands as tf32, true: fp16
// operand copies) and variant V (the handle uses the LeakyReLU / Dropout discriminator variants, whose epilogue code lives
// in separate instantiations; dW does not read V, so both variants share its kernels).  smem_attr is the max dynamic shared
// memory the kernel is cleared for (tc_plan_op).  The attribute is process-wide: a constant per instantiation, the largest
// tile any handle launches it with, never one op's own size.
enum TcRole { TC_FWD, TC_FWD_N, TC_FWD2, TC_DX, TC_DX_N, TC_DX2, TC_DW, TC_FWD_BIG, TC_DX_BIG, TC_DW_BIG, TC_ROLES };
struct TcKernel {
  void (*fn)(const TcOp*, FoldState*, int, AdamHyper, OperandMode);
  int threads, smem_attr;
};
constexpr int kTcSmemFwd = (int)tc_smem_bytes(256, TC_FWD_STAGES), kTcSmemDw = (int)tc_smem_bytes(128, TC_DW_STAGES);
template <bool F, bool V> const TcKernel kTcKernels[TC_ROLES] = {
    {k_gemm_tc<true, false, TC_FWD_STAGES, 256, 1, 8, 1, F, V>, TC_FWD_THREADS, kTcSmemFwd},
    {k_gemm_tc<true, false, TC_FWD_STAGES, 512, 1, 8, 1, F, V>, TC_FWD_THREADS, kTcSmemFwd},   // all 512 TMEM columns: room to park the epilogue's noise
    {k_gemm_tc<true, false, TC_FWD_STAGES, 512, 1, 8, 2, F, V>, TC_FWD_THREADS, kTcSmemMax},   // 256 features per CTA (layers >= 500 wide)
    {k_gemm_tc<false, false, TC_FWD_STAGES, 256, 1, 8, 1, F, V>, TC_FWD_THREADS, kTcSmemFwd},
    {k_gemm_tc<false, false, TC_FWD_STAGES, 512, 1, 8, 1, F, V>, TC_FWD_THREADS, kTcSmemFwd},
    {k_gemm_tc<false, false, TC_FWD_STAGES, 512, 1, 8, 2, F, V>, TC_FWD_THREADS, kTcSmemMax},
    {k_gemm_tc<true, true, TC_DW_STAGES, 128, 2, 4, 1, F, false>, TC_DW_THREADS, kTcSmemDw},
    {k_gemm_tc<true, false, TC_BIG_STAGES, 512, 1, 8, 2, F, V>, TC_FWD_THREADS, kTcSmemMax},
    {k_gemm_tc<false, false, TC_BIG_STAGES, 512, 1, 8, 2, F, V>, TC_FWD_THREADS, kTcSmemMax},
    {k_gemm_tc<true, true, TC_BIG_STAGES, 512, 1, 8, 2, F, false>, TC_FWD_THREADS, kTcSmemMax},
};
const TcKernel& tc_kernel(int role, bool f16, bool var) {
  static const TcKernel* const by_format[2][2] = {{kTcKernels<false, false>, kTcKernels<false, true>},
                                                  {kTcKernels<true, false>, kTcKernels<true, true>}};
  return by_format[f16][var][role];
}
bool tc_variant(const mrgan_handle* h) { return h->cfg.hidden_act != MRGAN_ACT_RELU || h->cfg.dropout > 0.0f; }

EncodeTiledFn tc_encoder() {
  EncodeTiledFn fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&fn, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess) return nullptr;
  return fn;
}

// Large-batch forward / dX (more than 256 stacked rows): batch rows per tile and feature sub-tiles per CTA.  256 x 256
// tiles are the efficient shape, but a narrow layer or a rank's slice of the batch leaves most of the 148 SMs without a
// tile (D layer 1 at 3072 local rows: 4 x 12 = 48 CTAs; the generator's dX over K = 12032: 2 x 4 = 8 CTAs, each alone on
// a 188-step contraction): fall back to 128-feature CTAs and then to narrower row tiles until the grid fills the chip.
void tc_pick_tile(int rows, int feats, int nf, int* bn, bool* mt1) {
  *bn = 256; *mt1 = false;
  auto tiles = [&](int b, bool one) { return ((feats + (one ? 127 : 255)) / (one ? 128 : 256)) * ((rows + b - 1) / b) * nf; };
  if (tiles(256, false) >= 120) return;
  *mt1 = true;
  for (int b : {256, 128, 64}) { *bn = b; if (tiles(b, true) >= 120) return; }
}

int tc_mode(const OpInfo& oi) { return oi.at ? 2 : (oi.bt ? 1 : 0); }   // 0 fwd, 1 dX, 2 dW

// Batch rows per tile (MMA-N) of one fold's GEMM; bn_big: those of a forward / dX with more than 256 rows (tc_pick_tile).
int tc_fold_bn(const GemmDesc& g, int mode, int bn_big) {
  if (mode == 2) return g.K > 512 ? 256 : 128;   // dW: a long contraction (large batch) is a regular big GEMM: 256 x 256 tiles
  return g.M <= 256 ? round_up(g.M, 16) : bn_big;
}

// fills the tcgen05 view of one GEMM (shapes in the fp32 path's convention)
// esz = 2: g.A / g.B point at fp16 operand copies (pitches in elements); the epilogue side of g is unchanged.
bool tc_fill_op(EncodeTiledFn fn, TcOp& t, const GemmDesc& g, int mode, int esz = 4, int bn_big = 256) {
  t.g = g;
  t.esz = esz;
  t.ME = g.N; t.NE = g.M; t.KE = g.K;
  t.bn = tc_fold_bn(g, mode, bn_big);
  const int kb = 128 / esz;   // contraction rows of an MN-major box = elements of one 128-byte row
  if (mode == 0)              // forward: C[M rows, N feats] = act[M, K] @ W[K, N]
    return make_map(fn, &t.mapA, g.B, g.N, g.K, g.ldb, kb, true, 0, esz) && make_map(fn, &t.mapB, g.A, g.K, g.M, g.lda, t.bn, false, 0, esz);
  if (mode == 1)              // dX: C[M rows, N in-feats] = dZ[M, K] @ W[N, K]^T
    return make_map(fn, &t.mapA, g.B, g.K, g.N, g.ldb, 128, false, 0, esz) && make_map(fn, &t.mapB, g.A, g.K, g.M, g.lda, t.bn, false, 0, esz);
  // dW: C[M in-feats(+1), N out-feats] = act[K rows, M]^T @ dZ[K rows, N]
  return make_map(fn, &t.mapA, g.B, g.N, g.K, g.ldb, kb, true, 0, esz) && make_map(fn, &t.mapB, g.A, g.M, g.K, g.lda, kb, true, 0, esz);
}

int tc_debug_gemm(mrgan_handle* h, int mode, const GemmDesc& g, int esz) {
  EncodeTiledFn fn = tc_encoder();
  if (!fn) return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  TcOp t; memset(&t, 0, sizeof(t));
  if (!tc_fill_op(fn, t, g, mode, esz)) return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  Temps tmp;
  TcOp* d = nullptr;
  CK(tmp.alloc(&d, sizeof(TcOp)));
  CK(cudaMemcpyAsync(d, &t, sizeof(t), cudaMemcpyHostToDevice, h->stream));
  const TcKernel& k = tc_kernel(mode == 0 ? TC_FWD : (mode == 1 ? TC_DX : TC_DW), esz == 2, tc_variant(h));
  CK(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, k.smem_attr));
  const dim3 grid((t.ME + 127) / 128, (t.NE + t.bn - 1) / t.bn, 1);
  const OperandMode om0{0, 1.0f, nullptr, nullptr};
  launch_k(h, k.fn, grid, k.threads, tc_smem_bytes(t.bn, mode == 2 ? TC_DW_STAGES : TC_FWD_STAGES), h->stream, (const TcOp*)d,
           h->d_folds, 0, h->hp, om0);
  CK(cudaStreamSynchronize(h->stream));
  return MRGAN_OK;
}

// The launch plan of one op: which k_gemm_tc instantiation runs it (or the fused dW+Adam kernel), on what grid and with
// how much shared memory, from the op's shapes over the folds, the precision and variant, the fused heads and the
// fused-Adam flag.  Clears the chosen kernel for its shared memory.  No-op for an unused op.
int tc_plan_op(mrgan_handle* h, int op) {
  const OpInfo& oi = h->ops[op];
  TcPlan& p = h->tc_plan[op];
  p = TcPlan();
  if (!oi.used) return MRGAN_OK;
  const int nf = h->nf, mode = tc_mode(oi);
  const bool f16 = h->om.mode == 2;
  bool mt1 = false;   // large-batch forward / dX whose 256 x 256 tiling would leave SMs idle: 128-feature CTAs
  if (mode != 2 && oi.maxM > 256) tc_pick_tile(oi.maxM, oi.maxN, nf, &p.bn_big, &mt1);
  for (int f = 0; f < nf; ++f) {
    const GemmDesc& g = h->h_descs[(size_t)op * nf + f];
    p.bn = std::max(p.bn, tc_fold_bn(g, mode, p.bn_big));
    p.maxME = std::max(p.maxME, g.N);
    p.maxNE = std::max(p.maxNE, g.M);
  }
  p.gx = (p.maxME + 127) / 128;
  // two feature sub-tiles per CTA when the layer is wide enough and the 4-stage ring still fits in 227 KB
  const bool mt2 = p.maxME >= 500 && tc_smem_bytes(p.bn, TC_FWD_STAGES, 2) <= kTcSmemMax;
  const bool head_mt2 = (h->tc_heads & 2) && op == OP_D5G;      // feature matching: one CTA sums the loss over all 250 features
  int role;
  if (p.bn == 256 && (oi.at || p.maxME >= 500) && !mt1) {     // large-batch regime
    role = mode == 0 ? TC_FWD_BIG : (mode == 1 ? TC_DX_BIG : TC_DW_BIG);
    p.gx = (p.maxME + 255) / 256;
    p.smem = tc_smem_bytes(256, TC_BIG_STAGES, 2);
    // Large-batch dW without the fused Adam: the narrow layers' gradients are a handful of 256x256 tiles with a contraction
    // of thousands of rows -> split the contraction over ~2 CTAs per SM, partial products to a workspace (tc_setup), summed
    // in slice order.
    if (oi.at && !h->tc_fused_adam) {
      const int kblk = f16 ? 64 : TC_KBLK;      // contraction rows per stage (one 128-byte row of operand elements)
      const int nkb = (h->h_descs[(size_t)op * nf].K + kblk - 1) / kblk;
      const int tiles = ((p.maxME + 255) / 256) * ((p.maxNE + 255) / 256) * nf;
      const int ks = std::min(std::min(2 * 148 / tiles, nkb / 8), 32);
      if (ks >= 2) {
        const int per = (nkb + ks - 1) / ks;
        p.ks = (nkb + per - 1) / per;           // no empty slice
      }
    }
  } else if (!oi.at && !mt1 && (mt2 || head_mt2)) {
    role = mode == 0 ? TC_FWD2 : TC_DX2;
    p.gx = (p.maxME + 255) / 256;
    p.smem = tc_smem_bytes(p.bn, TC_FWD_STAGES, 2);
  } else if (!oi.at) {
    // one CTA per SM anyway once the stages exceed half the shared memory: take the whole TMEM then (noise parking)
    p.smem = tc_smem_bytes(p.bn, TC_FWD_STAGES);
    const bool whole = 2 * p.smem > kTcSmemMax;
    role = mode == 0 ? (whole ? TC_FWD_N : TC_FWD) : (whole ? TC_DX_N : TC_DX);
  } else if (h->tc_fused_adam) {
    p.fused = true;
    if (f16) CK(cudaFuncSetAttribute(k_dw_adam_tc<true, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcAdamCfg<true, 32>::SMEM));
    else CK(cudaFuncSetAttribute(k_dw_adam_tc<false, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcAdamCfg<false, 16>::SMEM));
    return MRGAN_OK;
  } else {
    role = TC_DW;
    p.smem = tc_smem_bytes(p.bn, TC_DW_STAGES);
  }
  p.k = &tc_kernel(role, f16, tc_variant(h));
  CK(cudaFuncSetAttribute(p.k->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, p.k->smem_attr));
  return MRGAN_OK;
}

// f16 handles: the fp16 copy of an operand buffer, in the arena's shadow or in the generator workspace's own
const __half* half_copy(const mrgan_handle* h, const float* p) {
  const mrgan_handle::GenWork& G = h->gen;
  if (G.mem && p >= G.om.fbase && p < G.om.fbase + G.hfloats) return G.hmem + (p - G.om.fbase);
  return h->harena + (p - h->om.fbase);
}

// the launch plan of op and the tcgen05 views of its descriptors, one per fold (ts[0 .. nf)); no-op for an unused op
int tc_make_op(mrgan_handle* h, EncodeTiledFn fn, int op, TcOp* ts) {
  TRY(tc_plan_op(h, op));
  const OpInfo& oi = h->ops[op];
  if (!oi.used) return MRGAN_OK;
  const int nf = h->nf, mode = tc_mode(oi), bn_big = h->tc_plan[op].bn_big;
  for (int f = 0; f < nf; ++f) {
    const GemmDesc& g = h->h_descs[(size_t)op * nf + f];
    TcOp& t = ts[f];
    if (h->om.mode == 2) {    // operands come from the fp16 copies (same element offsets and pitches as the fp32 buffers)
      GemmDesc gh = g;
      gh.A = reinterpret_cast<const float*>(half_copy(h, g.A));
      gh.B = reinterpret_cast<const float*>(half_copy(h, g.B));
      if (!tc_fill_op(fn, t, gh, mode, 2, bn_big)) return fail(nullptr, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled (fp16 operands) failed");
      t.g = g;                // the epilogue keeps addressing the fp32 buffers (and derives the copies' addresses itself)
    } else if (!tc_fill_op(fn, t, g, mode, 4, bn_big)) return fail(nullptr, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    t.net = (op == OP_GW1 || op == OP_GW2 || op == OP_GW3) ? 1 : 0;
    if (h->tc_heads) {
      t.stats = h->d_step_stats + (size_t)f * 4;
      t.stats_stride = nf * 4;
      if (op == OP_D6 && (h->tc_heads & 1)) { t.head = HEAD_DISC; t.hd = h->d_loss + f; }
      else if (op == OP_D5G && (h->tc_heads & 2)) { t.head = HEAD_FM; t.hd = h->d_loss + f; }
      else if (op == OP_G1 && (h->tc_heads & 4)) { t.head = HEAD_BN; t.hd = h->d_bn + f; }
    }
  }
  return MRGAN_OK;
}

int tc_setup(mrgan_handle* h) {
  EncodeTiledFn fn = tc_encoder();
  if (!fn) return fail(nullptr, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  if (h->R > 512) h->tc_fused_adam = false;   // large batch: dW is tensor-bound -> big-tile GEMM + flat Adam instead of the fused kernel
  const int nf = h->nf;
  // reductions fused into GEMM epilogues: the reference batch regime (one batch tile, batch statistics local to the GPU).
  // BatchNorm backward stays the stand-alone k_bn_bwd: fused into GX2's epilogue it measured 1-2 % slower (a thread per
  // feature walks all 50 rows twice behind a GEMM whose own work is tiny).
  h->tc_heads = (h->cfg.model == MRGAN_MODEL_GAN && h->tc_fused_adam && !h->d_dpbufs && h->R <= 256 && h->cfg.n_classes <= 32) ? 7 : 0;
  std::vector<TcOp> ops((size_t)NUM_OPS * nf);
  memset(ops.data(), 0, ops.size() * sizeof(TcOp));
  for (int op = 0; op < NUM_OPS; ++op) {
    const int rc = tc_make_op(h, fn, op, &ops[(size_t)op * nf]);
    if (rc != MRGAN_OK) return rc;
  }
  // the split-K dW ops (tc_plan_op): the partial products of each contraction slice, laid out like C
  size_t ws_floats = 0;
  for (int op = 0; op < NUM_OPS; ++op)
    for (int f = 0; f < nf && h->tc_plan[op].ks > 1; ++f) {
      TcOp& t = ops[(size_t)op * nf + f];
      t.ws_stride = t.NE * t.g.ldc;
      t.ws = reinterpret_cast<float*>(ws_floats);     // offset now, pointer once the workspace exists
      ws_floats += (size_t)h->tc_plan[op].ks * t.ws_stride;
    }
  if (ws_floats) {
    if (cudaMalloc(&h->d_tcws, ws_floats * sizeof(float)) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMalloc split-K workspace");
    cudaMemset(h->d_tcws, 0, ws_floats * sizeof(float));      // pad columns are never written and must read as zero
    for (int op = 0; op < NUM_OPS; ++op)
      for (int f = 0; f < nf && h->tc_plan[op].ks > 1; ++f) {
        TcOp& t = ops[(size_t)op * nf + f];
        t.ws = h->d_tcws + reinterpret_cast<size_t>(t.ws);
      }
  }
  if (cudaMalloc(&h->d_tcops, ops.size() * sizeof(TcOp)) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMalloc tc ops");
  if (cudaMemcpy(h->d_tcops, ops.data(), ops.size() * sizeof(TcOp), cudaMemcpyHostToDevice) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMemcpy tc ops");
  if (h->tc_fused_adam) {
    std::vector<TcAdamOp> aops((size_t)NUM_OPS * nf);
    memset(aops.data(), 0, aops.size() * sizeof(TcAdamOp));
    for (int op = 0; op < NUM_OPS; ++op) {
      const OpInfo& oi = h->ops[op];
      if (!oi.used || !oi.at) continue;
      for (int f = 0; f < nf; ++f) {
        const TcOp& t = ops[(size_t)op * nf + f];
        TcAdamOp& a = aops[(size_t)op * nf + f];
        const GemmDesc& g = t.g;
        a.ME = t.ME; a.NE = t.NE; a.KE = t.KE; a.fold = g.fold; a.net = t.net;
        // operand boxes of 32 (fp16) / 16 (fp32) batch rows: 16 KB stages
        bool ok;
        if (h->om.mode == 2) {
          const __half* hA = h->harena + (g.A - h->om.fbase);
          const __half* hB = h->harena + (g.B - h->om.fbase);
          ok = make_map(fn, &a.mapA, hB, g.N, g.K, g.ldb, 32, true, 0, 2) && make_map(fn, &a.mapB, hA, g.M, g.K, g.lda, 32, true, 0, 2);
        } else {
          ok = make_map(fn, &a.mapA, g.B, g.N, g.K, g.ldb, 16, true) && make_map(fn, &a.mapB, g.A, g.M, g.K, g.lda, 16, true);
        }
        if (!ok) return fail(nullptr, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled (dW operands) failed");
        a.ginv = h->om.mode == 2 ? 1.0f / h->om.gscale : 1.0f;
        // the layer's weights and Adam slots: the gradient tensor's offset inside the flat buffers
        const size_t off = (size_t)(g.C - h->Gr);
        float *P = h->P + off, *Mo = h->Mo + off, *Vo = h->Vo + off;
        // fp16 operand copy of W (refreshed with every update), same geometry as the fp32 tensor
        if (h->om.mode == 2 && !make_map(fn, &a.mapH, h->harena + (P - h->om.fbase), t.ME, t.NE, g.ldc, TCA_KC, false, 128, 2))
          return fail(nullptr, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled (fp16 weight copy) failed");
        // W / m / v as [rows = in+1, cols = out] with the tensor's pitch; box 128 cols x KC rows, clipped at the logical extents
        if (!make_map(fn, &a.mapP, P, t.ME, t.NE, g.ldc, TCA_KC, false, 128) ||
            !make_map(fn, &a.mapM, Mo, t.ME, t.NE, g.ldc, TCA_KC, false, 128) ||
            !make_map(fn, &a.mapV, Vo, t.ME, t.NE, g.ldc, TCA_KC, false, 128))
          return fail(nullptr, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled (optimizer state) failed");
      }
    }
    if (cudaMalloc(&h->d_tcadam, aops.size() * sizeof(TcAdamOp)) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMalloc tc adam ops");
    if (cudaMemcpy(h->d_tcadam, aops.data(), aops.size() * sizeof(TcAdamOp), cudaMemcpyHostToDevice) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMemcpy tc adam ops");
  }
  // what is left for the flat Adam kernel when dW applies Adam itself
  std::vector<AdamRange> r0(nf), r1(nf);
  for (int f = 0; f < nf; ++f) {
    r0[f] = AdamRange{h->net[0][f].off, 0};
    if (h->cfg.model == MRGAN_MODEL_GAN) {
      const NetLayout& LG = h->net[1][f];
      r1[f] = AdamRange{LG.off + LG.t[1].off, LG.t[3].off - LG.t[1].off};     // gamma, beta (contiguous, padded)
    }
  }
  for (int n = 0; n < 2; ++n) {
    if (cudaMalloc(&h->d_ranges_tc[n], nf * sizeof(AdamRange)) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMalloc");
    if (cudaMemcpy(h->d_ranges_tc[n], (n == 0 ? r0 : r1).data(), nf * sizeof(AdamRange), cudaMemcpyHostToDevice) != cudaSuccess) return fail(nullptr, MRGAN_ERR_CUDA, "cudaMemcpy adam ranges");
  }
  return MRGAN_OK;
}

// the tcgen05 views of the ops [op0, op1) of a workspace, made on its first use -> dst [op1 - op0][nf]: the eval-backward ops
// (OP_EX*: mrgan_input_grad / mrgan_saliency) or the sample ops (OP_GG*, OP_S*: mrgan_generate / mrgan_sample_stats)
int tc_views(mrgan_handle* h, int op0, int op1, TcOp* dst) {
  EncodeTiledFn fn = tc_encoder();
  if (!fn) return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  std::vector<TcOp> ops((size_t)(op1 - op0) * h->nf);
  memset(ops.data(), 0, ops.size() * sizeof(TcOp));
  for (int op = op0; op < op1; ++op) {
    const int rc = tc_make_op(h, fn, op, &ops[(size_t)(op - op0) * h->nf]);
    if (rc != MRGAN_OK) return rc;
  }
  CK(cudaMemcpy(dst, ops.data(), ops.size() * sizeof(TcOp), cudaMemcpyHostToDevice));
  return MRGAN_OK;
}

void tc_teardown(mrgan_handle* h) {
  if (h->d_tcops) cudaFree(h->d_tcops);
  if (h->d_tcadam) cudaFree(h->d_tcadam);
  if (h->d_tcws) cudaFree(h->d_tcws);
  h->d_tcws = nullptr;
  for (int n = 0; n < 2; ++n) { if (h->d_ranges_tc[n]) cudaFree(h->d_ranges_tc[n]); h->d_ranges_tc[n] = nullptr; }
  for (int i = 0; i < NUM_OPS; ++i) h->tc_plan[i] = TcPlan();
  h->d_tcadam = nullptr;
  h->d_tcops = nullptr;
}

// dW + fused Adam of `nlayers` consecutive ops (op, op + 1, ...) of folds [f0, f0 + nfl) in ONE launch (grid.z = layer x fold;
// CTAs beyond a layer's extents exit at once)
void tc_launch_dw_adam(mrgan_handle* h, int op, int nlayers, int f0, int nfl, cudaStream_t st) {
  const bool f16 = h->om.mode == 2;
  int gx = 0, gy = 0;
  for (int l = 0; l < nlayers; ++l) {
    gx = std::max(gx, (h->tc_plan[op + l].maxME + 127) / 128);
    gy = std::max(gy, (h->tc_plan[op + l].maxNE + 127) / 128);
  }
  const dim3 grid(gx, gy, nlayers * nfl);
  const TcAdamOp* ad = h->d_tcadam + (size_t)op * h->nf + f0;
  if (f16) launch_k(h, k_dw_adam_tc<true, 32>, grid, dim3(192), TcAdamCfg<true, 32>::SMEM, st, ad, h->d_folds, h->hp, nfl, h->nf);
  else launch_k(h, k_dw_adam_tc<false, 16>, grid, dim3(192), TcAdamCfg<false, 16>::SMEM, st, ad, h->d_folds, h->hp, nfl, h->nf);
}

// one launch of op's plan over folds [f0, f0 + nfl); rows_override > 0: fewer batch rows (forward / dX)
void tc_launch_gemm(mrgan_handle* h, int op, int f0, int nfl, int rows_override, cudaStream_t st, const OperandMode& om) {
  const TcPlan& p = h->tc_plan[op];
  if (p.fused) { tc_launch_dw_adam(h, op, 1, f0, nfl, st); return; }
  const bool at = h->ops[op].at;
  const int NE = rows_override > 0 && !at ? rows_override : p.maxNE;
  const dim3 grid(p.gx, (NE + p.bn - 1) / p.bn, nfl * p.ks);
  const TcOp* d = (op < NUM_OPS ? h->d_tcops + (size_t)op * h->nf
                   : op < OP_GG1 ? h->sal.tcops + (size_t)(op - NUM_OPS) * h->nf : h->gen.tcops + (size_t)(op - OP_GG1) * h->nf) + f0;
  // dW kernels take the number of contraction slices in place of rows_override
  launch_k(h, p.k->fn, grid, p.k->threads, p.smem, st, d, h->d_folds, at ? p.ks : rows_override, h->hp, om);
  if (p.ks > 1) {
    const int n4 = p.maxNE * pitch8(p.maxME) / 4;
    launch_k(h, k_splitk_reduce, dim3(std::min((n4 + 255) / 256, 1184), nfl, 1), dim3(256), 0, st, d, p.ks);
  }
}

}  // namespace

// ====================================================================== C-ABI
extern "C" {

const char* mrgan_version(void) { return "mrgan-b200 0.2 (sm_100a)"; }

int mrgan_abi_info(int out[4]) {
  if (!out) return fail(nullptr, MRGAN_ERR_ARG, "abi_info: null pointer");
  out[0] = MRGAN_ABI_VERSION; out[1] = (int)sizeof(mrgan_config); out[2] = (int)sizeof(mrgan_fold_shape); out[3] = (int)sizeof(mrgan_epoch_stats);
  return MRGAN_OK;
}

int mrgan_default_config(int model, mrgan_config* cfg) {
  if (!cfg) return fail(nullptr, MRGAN_ERR_ARG, "cfg is null");
  memset(cfg, 0, sizeof(*cfg));
  cfg->model = model;
  cfg->n_folds = 1;
  cfg->n_classes = 6;
  cfg->noise_dim = 100;
  cfg->precision = MRGAN_PREC_FP32;
  cfg->shared_t = 1;
  cfg->eval_each_epoch = 1;
  cfg->device = 0;
  cfg->beta2 = 0.999f; cfg->adam_eps = 1e-8f; cfg->bn_eps = 2e-5f;
  cfg->unlabeled_weight = 1.0f; cfg->sigma_in = 0.3f; cfg->sigma_hidden = 0.5f;
  cfg->hidden_act = MRGAN_ACT_RELU; cfg->leaky_alpha = 0.3f; cfg->dropout = 0.0f;
  if (model == MRGAN_MODEL_NN) { cfg->batch = 20; cfg->lr = 1e-3f; cfg->beta1 = 0.9f; }
  else { cfg->batch = 50; cfg->lr = 6e-4f; cfg->beta1 = 0.5f; }
  return MRGAN_OK;
}

const char* mrgan_last_error(const mrgan_handle* h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int mrgan_create(const mrgan_config* cfg, const mrgan_fold_shape* folds, mrgan_handle** out) {
  mrgan_handle* h = nullptr;
  if (!cfg || !folds || !out) return fail(nullptr, MRGAN_ERR_ARG, "null argument");
  *out = nullptr;
  if (cfg->n_folds < 1 || cfg->batch < 1 || cfg->n_classes < 2 || cfg->n_classes > 64 || cfg->noise_dim < 1)
    return fail(nullptr, MRGAN_ERR_ARG, "bad config (n_folds/batch/n_classes/noise_dim)");
  if (cfg->model != MRGAN_MODEL_GAN && cfg->model != MRGAN_MODEL_NN && cfg->model != MRGAN_MODEL_SVM) return fail(nullptr, MRGAN_ERR_ARG, "bad model");
  if (cfg->model == MRGAN_MODEL_SVM && cfg->precision != MRGAN_PREC_FP32)
    return fail(nullptr, MRGAN_ERR_ARG, "bad config: the SVM has one arithmetic path (precision must be MRGAN_PREC_FP32)");
  if (cfg->batch > (1 << 16)) return fail(nullptr, MRGAN_ERR_ARG, "batch too large");
  if ((cfg->hidden_act != MRGAN_ACT_RELU && cfg->hidden_act != MRGAN_ACT_LEAKY_RELU) || !(cfg->dropout >= 0.0f && cfg->dropout < 1.0f))
    return fail(nullptr, MRGAN_ERR_ARG, "bad config (hidden_act / dropout)");
  for (int f = 0; f < cfg->n_folds; ++f) {
    if (folds[f].D < 1 || folds[f].n_train < cfg->batch || folds[f].n_test < 1)
      return fail(nullptr, MRGAN_ERR_ARG, "bad fold shape");
    if (folds[f].n_train != folds[0].n_train)
      return fail(nullptr, MRGAN_ERR_ARG, "all folds of a handle must have the same n_train");
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device >= ndev)
    return fail(nullptr, MRGAN_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10 || prop.minor != 0)
    return fail(nullptr, MRGAN_ERR_NO_DEVICE, "device is not sm_100 (B200): the library holds sm_100a code only and has no CPU fallback");
  if (cfg->precision < MRGAN_PREC_FP32 || cfg->precision > MRGAN_PREC_F16) return fail(nullptr, MRGAN_ERR_ARG, "bad config (precision)");
  h = new mrgan_handle();
  h->cfg = *cfg;
  h->nf = cfg->n_folds;
  h->R = cfg->model == MRGAN_MODEL_GAN ? 3 * cfg->batch : cfg->batch;
  h->n_train = folds[0].n_train;
  h->shapes.assign(folds, folds + h->nf);
  h->fb.resize(h->nf);
  h->hp = AdamHyper{cfg->lr, cfg->beta1, cfg->beta2, cfg->adam_eps, cfg->shared_t, cfg->batch, cfg->batch, 0,
                    cfg->unlabeled_weight, cfg->bn_eps, cfg->n_classes, 0,
                    cfg->hidden_act == MRGAN_ACT_LEAKY_RELU ? cfg->leaky_alpha : 0.0f, cfg->dropout, 1.0f / (1.0f - cfg->dropout)};
  int ne = h->R;
  for (int f = 0; f < h->nf; ++f) ne = folds[f].n_test > ne ? folds[f].n_test : ne;
  h->NE = ne;
  auto cleanup = [&](int code) { mrgan_destroy(h); return code; };
  if (cudaSetDevice(cfg->device) != cudaSuccess) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, "cudaSetDevice failed"));
  // flat parameter space: all D nets, then all G nets
  long long off = 0;
  for (int n = 0; n < (cfg->model == MRGAN_MODEL_GAN ? 2 : (cfg->model == MRGAN_MODEL_NN ? 1 : 0)); ++n) {
    h->net[n].resize(h->nf);
    for (int f = 0; f < h->nf; ++f) {
      NetLayout L = n == 0 ? layout_disc(folds[f].D, cfg->n_classes) : layout_gen(folds[f].D, cfg->noise_dim);
      L.off = off;
      off += L.n;
      h->net[n][f] = L;
    }
  }
  h->n_flat = off;
  Arena sizing;
  layout_buffers(h, sizing);
  h->arena_bytes = sizing.off + 256;
  cudaError_t e = cudaMalloc(&h->arena, h->arena_bytes);
  if (e != cudaSuccess) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, std::string("cudaMalloc arena: ") + cudaGetErrorString(e)));
  e = cudaMemset(h->arena, 0, h->arena_bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, std::string("cudaMemset: ") + cudaGetErrorString(e)));
  Arena real; real.base = h->arena;
  layout_buffers(h, real);
  h->om = OperandMode{cfg->precision, 1.0f, reinterpret_cast<const float*>(h->arena), nullptr};
  if (cfg->precision == MRGAN_PREC_F16) {      // operand copies: one __half per float of the arena, zero like the arena
    e = cudaMalloc(&h->harena, h->arena_bytes / 2);
    if (e == cudaSuccess) e = cudaMemset(h->harena, 0, h->arena_bytes / 2);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, std::string("cudaMalloc fp16 operand arena: ") + cudaGetErrorString(e)));
    h->om.hbase = h->harena;
    // gradient-side operands: fp16 times a loss scale (saturating; see OperandMode).  MRGAN_LOSS_SCALE overrides the default.
    h->om.gscale = MRGAN_F16_LOSS_SCALE;
    if (const char* ls = getenv("MRGAN_LOSS_SCALE")) { const float v = (float)atof(ls); if (v >= 1.0f) h->om.gscale = v; }
  }
  bool ok = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < 16 && ok; ++i) ok = cudaEventCreateWithFlags(&h->ev_pool[i], cudaEventDisableTiming) == cudaSuccess;
  {
    const char* env = getenv("MRGAN_CHAINS");
    int nch = env ? atoi(env) : (h->nf >= 32 ? 4 : (h->nf >= 8 ? 2 : 1));
    if (nch < 1) nch = 1;
    if (nch > kMaxChains) nch = kMaxChains;
    if (nch > h->nf) nch = h->nf;
    h->nchains = nch;
    h->cmain[0] = h->stream; h->cside[0] = h->side;
    for (int ch = 1; ch < nch && ok; ++ch) {
      ok = cudaStreamCreateWithFlags(&h->cmain[ch], cudaStreamNonBlocking) == cudaSuccess &&
           cudaStreamCreateWithFlags(&h->cside[ch], cudaStreamNonBlocking) == cudaSuccess;
    }
  }
  ok = ok && cudaEventCreate(&h->ev0) == cudaSuccess && cudaEventCreate(&h->ev1) == cudaSuccess;
  ok = ok && cudaMallocHost(&h->h_epoch_stats, (size_t)h->nf * 8 * sizeof(float)) == cudaSuccess;
  ok = ok && cudaMallocHost(&h->h_scratch, 64 * sizeof(float)) == cudaSuccess;
  for (int s = 0; s < 2 && ok; ++s) {
    ok = ok && cudaMallocHost(&h->h_idx_pinned[s], (size_t)h->nf * 3 * h->n_train * sizeof(int)) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->idx_free[s], cudaEventDisableTiming) == cudaSuccess;
  }
  if (!ok) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, "stream/event/pinned allocation failed"));
  if (cfg->model != MRGAN_MODEL_SVM) {
    const int rc = build_descs(h); if (rc != MRGAN_OK) return cleanup(rc);
    init_ones(h);
  } else {      // the confusion rows of an SVM fold: (y_test, voted class)
    std::vector<EvalDesc> ev(h->nf);
    for (int f = 0; f < h->nf; ++f) ev[f] = EvalDesc{nullptr, 0, h->fb[f].yte, folds[f].n_test, 0, nullptr, h->fb[f].pred};
    if (cudaMemcpy(h->d_eval, ev.data(), h->nf * sizeof(EvalDesc), cudaMemcpyHostToDevice) != cudaSuccess)
      return cleanup(fail(nullptr, MRGAN_ERR_CUDA, "create: descriptor upload failed"));
  }
  if (cfg->model == MRGAN_MODEL_GAN && cfg->batch > 256) {   // large batch: row-parallel split BatchNorm / feature-matching kernels
    int rc = alloc_split_bufs(h);
    if (rc != MRGAN_OK) return cleanup(rc);
  }
  if (cfg->precision != MRGAN_PREC_FP32) {
    h->tc_fused_adam = true;
    int rc = tc_setup(h);
    if (rc != MRGAN_OK) return cleanup(rc);
  }
  if (cfg->model == MRGAN_MODEL_GAN) {     // the device-side epoch permutations sort in shared memory
    e = cudaFuncSetAttribute(k_epoch_perm, cudaFuncAttributeMaxDynamicSharedMemorySize, PERM_MAX * 8);
    if (e != cudaSuccess) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, std::string("create: k_epoch_perm: ") + cudaGetErrorString(e)));
  }
  e = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return cleanup(fail(nullptr, MRGAN_ERR_CUDA, std::string("create: ") + cudaGetErrorString(e)));
  *out = h;
  return MRGAN_OK;
}

int mrgan_destroy(mrgan_handle* h) {
  if (!h) return MRGAN_OK;
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  drop_graphs(h);
  for (auto& ds : h->datasets) { if (ds.x) cudaFree(ds.x); if (ds.y) cudaFree(ds.y); }
  if (h->d_prep_stats) cudaFree(h->d_prep_stats);
  if (h->d_prep_rows) cudaFree(h->d_prep_rows);
  if (h->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->nccl_comm);
  if (!h->dp_virtual)
    for (int p = 0; p < DP_MAX_RANKS; ++p) {
      if (h->peer_arena[p] && h->peer_arena[p] != h->arena) cudaIpcCloseMemHandle(h->peer_arena[p]);
      if (h->peer_harena[p] && h->peer_harena[p] != h->harena) cudaIpcCloseMemHandle(h->peer_harena[p]);
    }
  if (h->d_dpmem) cudaFree(h->d_dpmem);
  if (h->d_dpbufs) cudaFree(h->d_dpbufs);
  if (h->sal.mem) cudaFree(h->sal.mem);
  gen_free(h);
  tc_teardown(h);
  if (h->svm.mem) cudaFree(h->svm.mem);
  if (h->svm.cv_mem) cudaFree(h->svm.cv_mem);
  if (h->arena) cudaFree(h->arena);
  if (h->harena) cudaFree(h->harena);
  if (h->h_epoch_stats) cudaFreeHost(h->h_epoch_stats);
  if (h->h_scratch) cudaFreeHost(h->h_scratch);
  for (int s = 0; s < 2; ++s) {
    if (h->h_idx_pinned[s]) cudaFreeHost(h->h_idx_pinned[s]);
    if (h->idx_free[s]) cudaEventDestroy(h->idx_free[s]);
  }
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (int i = 0; i < 16; ++i) if (h->ev_pool[i]) cudaEventDestroy(h->ev_pool[i]);
  for (int ch = 1; ch < kMaxChains; ++ch) { if (h->cmain[ch]) cudaStreamDestroy(h->cmain[ch]); if (h->cside[ch]) cudaStreamDestroy(h->cside[ch]); }
  if (h->side) cudaStreamDestroy(h->side);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return MRGAN_OK;
}

int mrgan_sync(mrgan_handle* h) {
  TRY(enter(h, "sync", 0));
  TRY(ready(h, "sync", 0));
  CK(cudaStreamSynchronize(h->stream));
  return MRGAN_OK;
}

int64_t mrgan_num_params(const mrgan_handle* h, int fold, int net) {
  if (!h || fold < 0 || fold >= h->nf || net < 0 || net > 1 || h->net[net].empty()) return -1;
  return h->net[net][fold].n_ref;
}

int mrgan_set_params(mrgan_handle* h, int fold, int net, const float* src, int64_t n) {
  TRY(enter(h, "set_params", FOLD | NETS, fold));
  if (net < 0 || net > 1 || h->net[net].empty()) return fail(h, MRGAN_ERR_ARG, "no such net in this model");
  const NetLayout& L = h->net[net][fold];
  if (!src || n != L.n_ref) return fail(h, MRGAN_ERR_ARG, "set_params: length does not match mrgan_num_params");
  TRY(ready(h, "set_params", FOLD | NETS, fold));
  std::vector<float> buf((size_t)L.n, 0.f);
  pack_params(h, fold, net, src, buf, true, nullptr);
  CK(cudaMemcpyAsync(h->P + L.off, buf.data(), (size_t)L.n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  // refresh the fp16 operand copy of the uploaded weights (the tf32 path reads the fp32 master weights unrounded)
  if (h->om.mode == 2) launch_k(h, k_to_half, 256, 256, 0, h->stream, h->P + L.off, (size_t)L.n, h->om);
  return complete(h);
}

static int get_flat(mrgan_handle* h, int fold, int net, const float* dev, float* dst, int64_t n) {
  const NetLayout& L = h->net[net][fold];
  if (!dst || n != L.n_ref) return fail(h, MRGAN_ERR_ARG, "length does not match mrgan_num_params");
  std::vector<float> buf((size_t)L.n);
  CK(cudaMemcpyAsync(buf.data(), dev + L.off, (size_t)L.n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  pack_params(h, fold, net, nullptr, buf, false, dst);
  return MRGAN_OK;
}

int mrgan_get_params(mrgan_handle* h, int fold, int net, float* dst, int64_t n) {
  TRY(enter(h, "get_params", FOLD | NETS, fold));
  if (net < 0 || net > 1 || h->net[net].empty()) return fail(h, MRGAN_ERR_ARG, "no such net in this model");
  TRY(ready(h, "get_params", FOLD | NETS, fold));
  return get_flat(h, fold, net, h->P, dst, n);
}

int mrgan_get_adam(mrgan_handle* h, int fold, int net, float* m, float* v, int64_t n) {
  TRY(enter(h, "get_adam", FOLD | NETS, fold));
  if (net < 0 || net > 1 || h->net[net].empty()) return fail(h, MRGAN_ERR_ARG, "no such net in this model");
  TRY(ready(h, "get_adam", FOLD | NETS, fold));
  TRY(get_flat(h, fold, net, h->Mo, m, n));
  return get_flat(h, fold, net, h->Vo, v, n);
}

int mrgan_get_counters(mrgan_handle* h, int fold, int* iterations, int* rng_step) {
  TRY(enter(h, "get_counters", FOLD | NETS, fold));
  TRY(ready(h, "get_counters", FOLD | NETS, fold));
  FoldState fs;
  CK(cudaMemcpyAsync(&fs, h->d_folds + fold, sizeof(fs), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (iterations) *iterations = h->cfg.shared_t ? fs.iterations : fs.it_net[0];
  if (rng_step) *rng_step = fs.rng_step;
  return MRGAN_OK;
}

// ------------------------------------------------------------------ checkpoint state (include/mrgan.h "Checkpoints")
int mrgan_set_adam(mrgan_handle* h, int fold, int net, const float* m, const float* v, int64_t n) {
  TRY(enter(h, "set_adam", FOLD | NETS, fold));
  if (net < 0 || net > 1 || h->net[net].empty()) return fail(h, MRGAN_ERR_ARG, "no such net in this model");
  const NetLayout& L = h->net[net][fold];
  if (!m || !v || n != L.n_ref) return fail(h, MRGAN_ERR_ARG, "set_adam: null pointer or length does not match mrgan_num_params");
  TRY(ready(h, "set_adam", FOLD | NETS | LOCAL, fold));
  std::vector<float> bm((size_t)L.n, 0.f), bv((size_t)L.n, 0.f);      // pad columns stay zero, as training leaves them
  pack_params(h, fold, net, m, bm, true, nullptr);
  pack_params(h, fold, net, v, bv, true, nullptr);
  CK(cudaMemcpyAsync(h->Mo + L.off, bm.data(), (size_t)L.n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->Vo + L.off, bv.data(), (size_t)L.n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  return complete(h);
}

// {iterations, it_net[0], it_net[1], rng_step}: four consecutive ints of FoldState, copied as one block
static_assert(offsetof(FoldState, it_net) == offsetof(FoldState, iterations) + sizeof(int) &&
              offsetof(FoldState, rng_step) == offsetof(FoldState, iterations) + 3 * sizeof(int), "FoldState counter block");

int mrgan_get_fold_counters(mrgan_handle* h, int fold, int32_t out[4]) {
  TRY(enter(h, "get_fold_counters", FOLD | NETS, fold));
  if (!out) return fail(h, MRGAN_ERR_ARG, "get_fold_counters: null pointer");
  TRY(ready(h, "get_fold_counters", FOLD | NETS | LOCAL, fold));
  CK(cudaMemcpyAsync(h->h_scratch, reinterpret_cast<const char*>(h->d_folds + fold) + offsetof(FoldState, iterations),
                     4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  memcpy(out, h->h_scratch, 4 * sizeof(int32_t));
  return MRGAN_OK;
}

int mrgan_set_fold_counters(mrgan_handle* h, int fold, const int32_t in[4]) {
  TRY(enter(h, "set_fold_counters", FOLD | NETS, fold));
  if (!in) return fail(h, MRGAN_ERR_ARG, "set_fold_counters: null pointer");
  for (int i = 0; i < 4; ++i)
    if (in[i] < 0) return fail(h, MRGAN_ERR_ARG, "set_fold_counters: negative counter");
  TRY(ready(h, "set_fold_counters", FOLD | NETS | LOCAL, fold));
  // lr_t is not part of the state: k_prep derives it from these counters at the start of every step
  memcpy(h->h_scratch, in, 4 * sizeof(int32_t));
  CK(cudaMemcpyAsync(reinterpret_cast<char*>(h->d_folds + fold) + offsetof(FoldState, iterations), h->h_scratch,
                     4 * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  return complete(h);
}

int mrgan_load_fold(mrgan_handle* h, int fold, const float* x_train, const int32_t* y_train, const float* x_test,
                    const int32_t* y_test) {
  TRY(enter(h, "load_fold", FOLD, fold));
  if (!x_train || !y_train || !x_test || !y_test) return fail(h, MRGAN_ERR_ARG, "load_fold: null pointer");
  const mrgan_fold_shape& s = h->shapes[fold];
  for (int i = 0; i < s.n_train; ++i)
    if (y_train[i] < 0 || y_train[i] >= h->cfg.n_classes) return fail(h, MRGAN_ERR_ARG, "load_fold: y_train label out of range");
  for (int i = 0; i < s.n_test; ++i)
    if (y_test[i] < 0 || y_test[i] >= h->cfg.n_classes) return fail(h, MRGAN_ERR_ARG, "load_fold: y_test label out of range");
  TRY(ready(h, "load_fold", FOLD, fold));
  FoldBuffers& b = h->fb[fold];
  const size_t w = (size_t)s.D * sizeof(float);
  CK(cudaMemcpy2DAsync(b.xtr, (size_t)pitch8(s.D) * sizeof(float), x_train, w, w, s.n_train, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpy2DAsync(b.xte, (size_t)b.lda[0] * sizeof(float), x_test, w, w, s.n_test, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(b.ytr, y_train, (size_t)s.n_train * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(b.yte, y_test, (size_t)s.n_test * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  to_operand(h, b.xte, (size_t)s.n_test * b.lda[0]);      // X_test feeds the first eval MMA directly (ones column included)
  TRY(complete(h));
  b.loaded = true;
  return MRGAN_OK;
}

int mrgan_load_dataset(mrgan_handle* h, int slot, const float* x, const int32_t* y, int n_rows, int D) {
  TRY(enter(h, "load_dataset", 0));
  if (slot < 0 || slot >= 8 || !x || !y || n_rows < 1 || D < 1) return fail(h, MRGAN_ERR_ARG, "load_dataset: bad argument");
  for (int i = 0; i < n_rows; ++i)
    if (y[i] < 0 || y[i] >= h->cfg.n_classes) return fail(h, MRGAN_ERR_ARG, "load_dataset: label out of range");
  TRY(ready(h, "load_dataset", 0));
  mrgan_handle::Dataset& ds = h->datasets[slot];
  if (ds.x && (ds.n != n_rows || ds.D != D)) { cudaFree(ds.x); cudaFree(ds.y); ds.x = nullptr; ds.y = nullptr; }
  ds.n = n_rows; ds.D = D; ds.ld = pitch8(D);
  if (!ds.x) {       // a re-upload of the same shape reuses the buffers (cudaFree / cudaMalloc synchronise the device)
    CK(cudaMalloc(&ds.x, (size_t)n_rows * ds.ld * sizeof(float)));
    CK(cudaMalloc(&ds.y, (size_t)n_rows * sizeof(int)));
  }
  CK(cudaMemcpy2DAsync(ds.x, (size_t)ds.ld * sizeof(float), x, (size_t)D * sizeof(float), (size_t)D * sizeof(float), n_rows,
                       cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(ds.y, y, (size_t)n_rows * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  return complete(h);
}

int mrgan_prepare_fold(mrgan_handle* h, int fold, int slot, const int32_t* train_rows, const int32_t* test_rows) {
  TRY(enter(h, "prepare_fold", FOLD, fold));
  if (slot < 0 || slot >= 8 || !h->datasets[slot].x) return fail(h, MRGAN_ERR_STATE, "prepare_fold: dataset slot is empty");
  if (!train_rows || !test_rows) return fail(h, MRGAN_ERR_ARG, "prepare_fold: null pointer");
  const mrgan_handle::Dataset& ds = h->datasets[slot];
  const mrgan_fold_shape& s = h->shapes[fold];
  if (ds.D != s.D) return fail(h, MRGAN_ERR_ARG, "prepare_fold: dataset width differs from the fold's D");
  for (int i = 0; i < s.n_train; ++i) if ((unsigned)train_rows[i] >= (unsigned)ds.n) return fail(h, MRGAN_ERR_ARG, "prepare_fold: train row out of range");
  for (int i = 0; i < s.n_test; ++i) if ((unsigned)test_rows[i] >= (unsigned)ds.n) return fail(h, MRGAN_ERR_ARG, "prepare_fold: test row out of range");
  TRY(ready(h, "prepare_fold", FOLD, fold));
  const int nrows = s.n_train + s.n_test;
  if (nrows > h->prep_rows_cap) {
    if (h->d_prep_rows) cudaFree(h->d_prep_rows);
    CK(cudaMalloc(&h->d_prep_rows, (size_t)nrows * sizeof(int)));
    h->prep_rows_cap = nrows;
  }
  if (2 * s.D > h->prep_stats_cap) {      // per-slice partial column sums: [PREP_SLICES][2 * D] doubles
    if (h->d_prep_stats) cudaFree(h->d_prep_stats);
    CK(cudaMalloc(&h->d_prep_stats, (size_t)PREP_SLICES * 2 * s.D * sizeof(double)));
    h->prep_stats_cap = 2 * s.D;
  }
  FoldBuffers& b = h->fb[fold];
  CK(cudaMemcpyAsync(h->d_prep_rows, train_rows, (size_t)s.n_train * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_prep_rows + s.n_train, test_rows, (size_t)s.n_test * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  const int gx = (s.D + 127) / 128;
  launch_k(h, k_col_stats, dim3(gx, PREP_SLICES), 128, 0, h->stream, ds.x, ds.ld, h->d_prep_rows, s.n_train, s.D, h->d_prep_stats);
  launch_k(h, k_scale_gather, dim3(gx, 64), 128, 0, h->stream, ds.x, ds.ld, h->d_prep_rows, s.n_train, s.D, h->d_prep_stats, PREP_SLICES,
           s.n_train, b.xtr, pitch8(s.D), ds.y, b.ytr, OperandMode{0, 1.0f, nullptr, nullptr});
  launch_k(h, k_scale_gather, dim3(gx, 64), 128, 0, h->stream, ds.x, ds.ld, h->d_prep_rows + s.n_train, s.n_test, s.D, h->d_prep_stats,
           PREP_SLICES, s.n_train, b.xte, b.lda[0], ds.y, b.yte, h->om);
  TRY(complete(h));     // the pageable index arrays are borrowed only for the call
  b.loaded = true;
  return MRGAN_OK;
}

int mrgan_disc_step(mrgan_handle* h, int fold, const float* x_lab, const int32_t* labels, const float* x_unl,
                    const float* z, float out[3]) {
  TRY(enter(h, "disc_step", FOLD | GAN, fold));
  if (!x_lab || !labels || !x_unl || !z || !out) return fail(h, MRGAN_ERR_ARG, "disc_step: null pointer");
  const int B = h->cfg.batch, D = h->shapes[fold].D, nd = h->cfg.noise_dim;
  for (int i = 0; i < B; ++i)
    if (labels[i] < 0 || labels[i] >= h->cfg.n_classes) return fail(h, MRGAN_ERR_ARG, "disc_step: label out of range");
  TRY(ready(h, "disc_step", FOLD | GAN | NOT_VIRTUAL, fold));
  FoldBuffers& b = h->fb[fold];
  const size_t w = (size_t)D * sizeof(float), ld = (size_t)pitch8(D) * sizeof(float);
  CK(cudaMemcpy2DAsync(b.stage_x, ld, x_lab, w, w, B, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpy2DAsync(b.stage_x + (size_t)B * pitch8(D), ld, x_unl, w, w, B, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(b.stage_y, labels, (size_t)B * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(b.stage_z, z, (size_t)B * nd * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  enqueue_disc_step(h, fold, 1, 0, 1);
  CK(cudaMemcpyAsync(h->h_scratch, h->d_step_stats + (size_t)fold * 4, 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  out[0] = h->h_scratch[0]; out[1] = h->h_scratch[1]; out[2] = h->h_scratch[2];
  return MRGAN_OK;
}

int mrgan_gen_step(mrgan_handle* h, int fold, const float* x_unl, const float* z, float out[1]) {
  TRY(enter(h, "gen_step", FOLD | GAN, fold));
  if (!x_unl || !z || !out) return fail(h, MRGAN_ERR_ARG, "gen_step: null pointer");
  TRY(ready(h, "gen_step", FOLD | GAN | NOT_VIRTUAL, fold));
  const int B = h->cfg.batch, D = h->shapes[fold].D, nd = h->cfg.noise_dim;
  FoldBuffers& b = h->fb[fold];
  const size_t w = (size_t)D * sizeof(float), ld = (size_t)pitch8(D) * sizeof(float);
  CK(cudaMemcpy2DAsync(b.stage_x + (size_t)B * pitch8(D), ld, x_unl, w, w, B, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(b.stage_z, z, (size_t)B * nd * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  enqueue_gen_step(h, fold, 1, 0, 1);
  CK(cudaMemcpyAsync(h->h_scratch, h->d_step_stats + (size_t)fold * 4, 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  out[0] = h->h_scratch[3];
  return MRGAN_OK;
}

int mrgan_test_batch(mrgan_handle* h, int fold, const float* x, const int32_t* y, int n, float* err) {
  TRY(enter(h, "test_batch", FOLD | NETS, fold));
  if (!x || !y || !err) return fail(h, MRGAN_ERR_ARG, "test_batch: null pointer");
  if (n < 1 || n > h->NE) return fail(h, MRGAN_ERR_ARG, "test_batch: n exceeds max(n_test, rows of a train step)");
  for (int i = 0; i < n; ++i)
    if (y[i] < 0 || y[i] >= h->cfg.n_classes) return fail(h, MRGAN_ERR_ARG, "test_batch: label out of range");
  TRY(ready(h, "test_batch", FOLD | NETS, fold));
  FoldBuffers& b = h->fb[fold];
  TRY(stage_rows(h, fold, x, n));
  CK(cudaMemcpyAsync(b.ey_stage, y, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  enqueue_eval(h, fold, 1, true, n);
  CK(cudaMemcpyAsync(h->h_scratch, b.eval_out_s, 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  err[0] = h->h_scratch[1];
  return MRGAN_OK;
}

int mrgan_eval(mrgan_handle* h, int fold, float* err) {
  TRY(enter(h, "eval", FOLD | NETS, fold));
  if (!err) return fail(h, MRGAN_ERR_ARG, "eval: null pointer");
  TRY(ready(h, "eval", FOLD | NETS | LOADED, fold));
  enqueue_eval(h, fold, 1, false, 0);
  CK(cudaMemcpyAsync(h->h_scratch, h->fb[fold].eval_out, 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  err[0] = h->h_scratch[1];
  return MRGAN_OK;
}

int mrgan_epoch_result(mrgan_handle* h, mrgan_epoch_stats* stats) {
  TRY(enter(h, "epoch_result", NETS));
  TRY(ready(h, "epoch_result", NETS));
  CKS();
  if (stats)
    for (int f = 0; f < h->nf; ++f) {
      const float* s = h->h_epoch_stats + (size_t)f * 8;
      stats[f] = mrgan_epoch_stats{s[0], s[1], s[2], s[3], s[4]};
    }
  return MRGAN_OK;
}

int mrgan_set_epoch_rows(mrgan_handle* h, int fold, const int32_t* lab_rows, int n_lab, const int32_t* unl_rows, int n_unl) {
  TRY(enter(h, "set_epoch_rows", FOLD | GAN, fold));
  const int N = h->n_train;
  if (!lab_rows || n_lab < 1 || n_lab > N || n_lab > PERM_MAX) return fail(h, MRGAN_ERR_ARG, "set_epoch_rows: 1 <= n_lab <= min(n_train, 8192)");
  if (unl_rows ? (n_unl < 1 || n_unl > N || n_unl > PERM_MAX) : (n_unl != 0 || N > PERM_MAX))
    return fail(h, MRGAN_ERR_ARG, "set_epoch_rows: unlabeled subset must have 1..min(n_train, 8192) rows (none: n_train <= 8192)");
  for (int i = 0; i < n_lab; ++i) if ((unsigned)lab_rows[i] >= (unsigned)N) return fail(h, MRGAN_ERR_ARG, "set_epoch_rows: labeled row out of range");
  for (int i = 0; i < n_unl; ++i) if ((unsigned)unl_rows[i] >= (unsigned)N) return fail(h, MRGAN_ERR_ARG, "set_epoch_rows: unlabeled row out of range");
  TRY(ready(h, "set_epoch_rows", FOLD | GAN, fold));
  FoldBuffers& b = h->fb[fold];
  CK(cudaMemcpyAsync(b.lab_rows, lab_rows, (size_t)n_lab * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  if (unl_rows) CK(cudaMemcpyAsync(b.unl_rows, unl_rows, (size_t)n_unl * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  b.n_lab = n_lab; b.n_unl = unl_rows ? n_unl : 0;
  PermDesc pd{b.lab_rows, unl_rows ? b.unl_rows : nullptr, b.idx, n_lab, b.n_unl, N,
              (uint32_t)(h->shapes[fold].seed & 0xFFFFFFFFull), (uint32_t)(h->shapes[fold].seed >> 32)};
  CK(cudaMemcpyAsync(h->d_perm + fold, &pd, sizeof(pd), cudaMemcpyHostToDevice, h->stream));
  return complete(h);       // the pageable row arrays are borrowed only for the call
}

static int launch_epoch(mrgan_handle* h, int nb, mrgan_epoch_stats* stats);

int mrgan_train_epoch_seeded(mrgan_handle* h, uint32_t epoch, mrgan_epoch_stats* stats) {
  TRY(enter(h, "train_epoch_seeded", GAN));
  TRY(ready(h, "train_epoch_seeded", GAN | LOADED));
  for (int f = 0; f < h->nf; ++f)
    if (h->fb[f].n_lab < 1) return fail(h, MRGAN_ERR_STATE, "train_epoch_seeded before mrgan_set_epoch_rows");
  launch_k(h, k_epoch_perm, dim3(3, h->nf), 1024, PERM_MAX * 8, h->stream, h->d_perm, epoch);
  return launch_epoch(h, h->n_train / h->cfg.batch, stats);
}

int mrgan_debug_epoch_indices(mrgan_handle* h, int fold, int32_t* dst) {
  TRY(enter(h, "debug_epoch_indices", FOLD | NETS, fold));
  if (!dst) return fail(h, MRGAN_ERR_ARG, "debug_epoch_indices: null pointer");
  TRY(ready(h, "debug_epoch_indices", FOLD | NETS, fold));
  CK(cudaMemcpyAsync(dst, h->fb[fold].idx, (size_t)3 * h->n_train * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

int mrgan_train_epoch(mrgan_handle* h, const int32_t* idx_lab, const int32_t* idx_unl, const int32_t* idx_unl2,
                      mrgan_epoch_stats* stats) {
  TRY(enter(h, "train_epoch", GAN));
  if (!idx_lab || !idx_unl || !idx_unl2) return fail(h, MRGAN_ERR_ARG, "train_epoch: null index array");
  const size_t tot = (size_t)h->nf * h->n_train;
  for (size_t i = 0; i < tot; ++i)
    if ((unsigned)idx_lab[i] >= (unsigned)h->n_train || (unsigned)idx_unl[i] >= (unsigned)h->n_train ||
        (unsigned)idx_unl2[i] >= (unsigned)h->n_train)
      return fail(h, MRGAN_ERR_ARG, "train_epoch: row index out of range");
  TRY(ready(h, "train_epoch", GAN | LOADED));
  const int32_t* streams[3] = {idx_lab, idx_unl, idx_unl2};
  TRY(upload_indices(h, streams, 3, h->n_train));
  return launch_epoch(h, h->n_train / h->cfg.batch, stats);
}

// the epoch itself (index arrays already on their way on the handle's stream): one graph launch.  Data-parallel epochs are
// captured like the others (NCCL collectives and the fused exchange are stream-ordered graph nodes; one chain, so every
// rank issues them in the same order).
static int launch_epoch(mrgan_handle* h, int nb, mrgan_epoch_stats* stats) {
  TRY(build_graph(h, nb, nb));
  CK(cudaEventRecord(h->ev0, h->stream));
  CK(cudaGraphLaunch(h->graphs[nb], h->stream));
  h->launches += h->graph_nodes[nb];
  CK(cudaEventRecord(h->ev1, h->stream));
  h->epoch_pending = true;
  TRY(take_sticky(h));
  if (stats) return mrgan_epoch_result(h, stats);
  return MRGAN_OK;
}

int mrnn_step(mrgan_handle* h, int fold, const float* x, const int32_t* labels, int n, float out[2]) {
  TRY(enter(h, "mrnn_step", FOLD | NN, fold));
  if (!x || !labels || !out) return fail(h, MRGAN_ERR_ARG, "mrnn_step: null pointer");
  if (n < 1 || n > h->cfg.batch) return fail(h, MRGAN_ERR_ARG, "mrnn_step: n must be in [1, batch]");
  for (int i = 0; i < n; ++i)
    if (labels[i] < 0 || labels[i] >= h->cfg.n_classes) return fail(h, MRGAN_ERR_ARG, "mrnn_step: label out of range");
  TRY(ready(h, "mrnn_step", FOLD | NN, fold));
  FoldBuffers& b = h->fb[fold];
  const int D = h->shapes[fold].D;
  const size_t w = (size_t)D * sizeof(float);
  CK(cudaMemcpy2DAsync(b.stage_x, (size_t)pitch8(D) * sizeof(float), x, w, w, n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(b.stage_y, labels, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  enqueue_nn_step(h, fold, 1, 0, 1, n);
  CK(cudaMemcpyAsync(h->h_scratch, h->d_step_stats + (size_t)fold * 4, 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  out[0] = h->h_scratch[0]; out[1] = h->h_scratch[1];
  return MRGAN_OK;
}

int mrnn_train_epoch(mrgan_handle* h, const int32_t* idx, int n_idx, float* loss_acc) {
  TRY(enter(h, "mrnn_train_epoch", NN));
  if (!idx || n_idx < h->cfg.batch || n_idx > h->n_train || n_idx % h->cfg.batch)
    return fail(h, MRGAN_ERR_ARG, "mrnn_train_epoch: n_idx must be a multiple of batch in [batch, n_train]");
  for (size_t i = 0; i < (size_t)h->nf * n_idx; ++i)
    if ((unsigned)idx[i] >= (unsigned)h->n_train) return fail(h, MRGAN_ERR_ARG, "mrnn_train_epoch: row index out of range");
  TRY(ready(h, "mrnn_train_epoch", NN | LOADED));
  const int32_t* streams[1] = {idx};
  TRY(upload_indices(h, streams, 1, n_idx));
  TRY(launch_epoch(h, n_idx / h->cfg.batch, nullptr));
  if (loss_acc) {
    TRY(finish_pending(h));
    CKS();
    for (int f = 0; f < h->nf; ++f) { loss_acc[2 * f] = h->h_epoch_stats[f * 8]; loss_acc[2 * f + 1] = h->h_epoch_stats[f * 8 + 1]; }
  }
  return MRGAN_OK;
}

int mrnn_evaluate(mrgan_handle* h, int fold, float out[2]) {
  TRY(enter(h, "evaluate", FOLD | NETS, fold));
  if (!out) return fail(h, MRGAN_ERR_ARG, "evaluate: null pointer");
  TRY(ready(h, "evaluate", FOLD | NETS | LOADED, fold));
  enqueue_eval(h, fold, 1, false, 0);
  CK(cudaMemcpyAsync(h->h_scratch, h->fb[fold].eval_out, 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  out[0] = h->h_scratch[2]; out[1] = 1.0f - h->h_scratch[1];
  return MRGAN_OK;
}

int mrgan_fill_normal(mrgan_handle* h, int fold, int step, int tensor_id, int rows, int cols, int row0, float* dst) {
  TRY(enter(h, "fill_normal", FOLD | NETS, fold));
  if (!dst || rows < 1 || cols < 1) return fail(h, MRGAN_ERR_ARG, "fill_normal: bad argument");
  TRY(ready(h, "fill_normal", FOLD | NETS, fold));
  Temps tmp;
  float* d = nullptr;
  const size_t n = (size_t)rows * cols;
  CK(tmp.alloc(&d, n * sizeof(float)));
  launch_k(h, k_fill_normal, (unsigned)((n + 255) / 256), 256, 0, h->stream, d, h->d_folds, fold, step, tensor_id, rows, cols, row0);
  CK(cudaMemcpyAsync(dst, d, n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

int mrgan_adam_flat(mrgan_handle* h, float* p, float* m, float* v, const float* g, int64_t n, int t) {
  TRY(enter(h, "adam_flat", NETS));
  if (!p || !m || !v || !g || n < 1 || t < 1) return fail(h, MRGAN_ERR_ARG, "adam_flat: bad argument");
  TRY(ready(h, "adam_flat", NETS));
  const int64_t n4 = (n + 3) / 4;
  Temps tmp;
  float* d = nullptr;
  CK(tmp.alloc(&d, (size_t)n4 * 16 * 4));
  CK(cudaMemsetAsync(d, 0, (size_t)n4 * 16 * 4, h->stream));
  float *dp = d, *dm = d + n4 * 4, *dv = d + n4 * 8, *dg = d + n4 * 12;
  CK(cudaMemcpyAsync(dp, p, n * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(dm, m, n * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(dv, v, n * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(dg, g, n * 4, cudaMemcpyHostToDevice, h->stream));
  const double b1t = pow((double)h->hp.b1, (double)t), b2t = pow((double)h->hp.b2, (double)t);
  const float lr_t = (float)((double)h->hp.lr * sqrt(1.0 - b2t) / (1.0 - b1t));
  int blocks = (int)((n4 + 255) / 256); if (blocks > 4096) blocks = 4096;
  launch_k(h, k_adam_plain, blocks, 256, 0, h->stream, (float4*)dp, (float4*)dm, (float4*)dv, (const float4*)dg, n4, lr_t,
           h->hp.b1, h->hp.b2, h->hp.eps);
  CK(cudaMemcpyAsync(p, dp, n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(m, dm, n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(v, dv, n * 4, cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

static void svm_launch(mrgan_handle* h, int phase);

int mrgan_time_op(mrgan_handle* h, int which, int reps, float* ms_avg) {
  TRY(enter(h, "time_op", 0));
  if (!ms_avg || reps < 1) return fail(h, MRGAN_ERR_ARG, "time_op: bad argument");
  const bool svm = h->cfg.model == MRGAN_MODEL_SVM, gan = h->cfg.model == MRGAN_MODEL_GAN;
  if (svm != (which >= MRGAN_TIME_SVM_KMAT && which <= MRGAN_TIME_SVM_PREDICT))
    return fail(h, which < 0 || which > MRGAN_TIME_SAMPLE_STATS ? MRGAN_ERR_ARG : MRGAN_ERR_STATE, "time_op: op does not exist for this model");
  if (which < 0 || which > MRGAN_TIME_SAMPLE_STATS) return fail(h, MRGAN_ERR_ARG, "time_op: unknown op");
  if (!gan && (which == MRGAN_TIME_ADAM_G || which == MRGAN_TIME_GEN_STEP || which == MRGAN_TIME_DX1 || which == MRGAN_TIME_SAMPLE_STATS))
    return fail(h, MRGAN_ERR_STATE, "time_op: no generator in this model");
  const bool ro = which == MRGAN_TIME_SALIENCY || which == MRGAN_TIME_SAMPLE_STATS;
  TRY(ready(h, "time_op", svm ? FITTED : (LOADED | (ro ? LOCAL : 0u))));
  if (svm) return time_reps(h, reps, [&]() { svm_launch(h, which); }, ms_avg);
  if (which == MRGAN_TIME_SALIENCY) TRY(saliency_setup(h));
  if (which == MRGAN_TIME_SAMPLE_STATS) TRY(gen_setup(h));
  return time_reps(h, reps, [&]() {
    switch (which) {
      case MRGAN_TIME_ADAM_D: launch_adam(h, 0, h->nf, 0); break;
      case MRGAN_TIME_ADAM_G: launch_adam(h, 0, h->nf, 1); break;
      case MRGAN_TIME_DW1: launch_gemm(h, OP_DW1, 0, h->nf, 0); break;
      case MRGAN_TIME_FWD1: launch_gemm(h, OP_D1, 0, h->nf, 0); break;
      case MRGAN_TIME_DISC_STEP: if (gan) enqueue_disc_step(h, 0, h->nf, 0, 0); else enqueue_nn_step(h, 0, h->nf, 0, 0, h->cfg.batch); break;
      case MRGAN_TIME_GEN_STEP: enqueue_gen_step(h, 0, h->nf, 0, 0); break;
      case MRGAN_TIME_DX1: launch_gemm(h, OP_DX1G, 0, h->nf, 0); break;
      case MRGAN_TIME_SALIENCY: enqueue_saliency(h); break;
      case MRGAN_TIME_SAMPLE_STATS: enqueue_sample_stats(h, h->gen.NG, 0); break;
      default: break;
    }
  }, ms_avg);
}

int mrgan_nccl_unique_id(void* id128) {
  if (!id128) return fail(nullptr, MRGAN_ERR_ARG, "nccl_unique_id: null pointer");
  if (!nccl_load()) return fail(nullptr, MRGAN_ERR_STATE, "libnccl.so.2 not found");
  NcclId id;
  const int rc = g_nccl.GetUniqueId(&id);
  if (rc != 0) return fail(nullptr, MRGAN_ERR_CUDA, "ncclGetUniqueId failed");
  memcpy(id128, id.b, 128);
  return MRGAN_OK;
}

int mrgan_dp_init(mrgan_handle* h, int rank, int world, const void* id128) {
  TRY(enter(h, "dp_init", GAN));
  if (world < 1 || rank < 0 || rank >= world || !id128) return fail(h, MRGAN_ERR_ARG, "dp_init: bad rank / world / id");
  if (world > DP_MAX_RANKS) return fail(h, MRGAN_ERR_ARG, "dp_init: at most 8 ranks (one NVSwitch domain)");
  if (h->dp_world > 1 || h->nccl_comm) return fail(h, MRGAN_ERR_STATE, "dp_init called twice");
  if (world == 1) return MRGAN_OK;
  if (h->cfg.batch % 4) return fail(h, MRGAN_ERR_ARG, "dp_init: the local batch must be a multiple of 4 (noise row groups)");
  if (!nccl_load()) return fail(h, MRGAN_ERR_STATE, "libnccl.so.2 not found");
  TRY(ready(h, "dp_init", GAN));
  NcclId id; memcpy(id.b, id128, 128);
  const int nrc = g_nccl.CommInitRank(&h->nccl_comm, world, id, rank);
  if (nrc != 0) return fail(h, MRGAN_ERR_CUDA, std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(nrc) : "error"));
  return dp_switch(h, world, rank);
}

int mrgan_dp_ipc_export(mrgan_handle* h, void* out128) {
  TRY(enter(h, "dp_ipc_export", 0));
  if (!out128) return fail(h, MRGAN_ERR_ARG, "dp_ipc_export: null argument");
  TRY(ready(h, "dp_ipc_export", 0));
  memset(out128, 0, 128);
  cudaIpcMemHandle_t a;
  CK(cudaIpcGetMemHandle(&a, h->arena));
  memcpy(out128, &a, sizeof(a));
  if (h->harena) {
    CK(cudaIpcGetMemHandle(&a, h->harena));
    memcpy(static_cast<char*>(out128) + 64, &a, sizeof(a));
  }
  return MRGAN_OK;
}

int mrgan_dp_ipc_open(mrgan_handle* h, const void* handles, int world) {
  TRY(enter(h, "dp_ipc_open", 0));
  if (!handles) return fail(h, MRGAN_ERR_ARG, "dp_ipc_open: null argument");
  if (h->dp_world != world || world < 2 || world > DP_MAX_RANKS || h->dp_virtual)
    return fail(h, MRGAN_ERR_STATE, "dp_ipc_open: call after mrgan_dp_init with the same world size (at most 8 ranks)");
  TRY(ready(h, "dp_ipc_open", 0));
  const char* hb = static_cast<const char*>(handles);
  for (int p = 0; p < world; ++p) {
    if (p == h->dp_rank) { h->peer_arena[p] = h->arena; h->peer_harena[p] = h->harena; continue; }
    cudaIpcMemHandle_t a;
    memcpy(&a, hb + (size_t)p * 128, sizeof(a));
    void* ptr = nullptr;
    CK(cudaIpcOpenMemHandle(&ptr, a, cudaIpcMemLazyEnablePeerAccess));
    h->peer_arena[p] = static_cast<char*>(ptr);
    if (h->harena) {
      memcpy(&a, hb + (size_t)p * 128 + 64, sizeof(a));
      CK(cudaIpcOpenMemHandle(&ptr, a, cudaIpcMemLazyEnablePeerAccess));
      h->peer_harena[p] = static_cast<__half*>(ptr);
    }
  }
  h->dp_fused = true;
  dp_build_peers(h);
  drop_graphs(h);
  return MRGAN_OK;
}

int mrgan_dp_init_virtual(mrgan_handle* h, int world) {
  TRY(enter(h, "dp_init_virtual", GAN));
  if (h->dp_world > 1 || h->nccl_comm) return fail(h, MRGAN_ERR_STATE, "dp_init called twice");
  if (world < 2 || world != h->nf) return fail(h, MRGAN_ERR_ARG, "dp_init_virtual: the handle must hold exactly `world` folds (one per virtual rank)");
  if (world > DP_MAX_RANKS) return fail(h, MRGAN_ERR_ARG, "dp_init_virtual: at most 8 ranks");
  if (h->cfg.batch % 4) return fail(h, MRGAN_ERR_ARG, "dp_init_virtual: the local batch must be a multiple of 4 (noise row groups)");
  for (int f = 1; f < h->nf; ++f)
    if (h->shapes[f].D != h->shapes[0].D || h->shapes[f].seed != h->shapes[0].seed)
      return fail(h, MRGAN_ERR_ARG, "dp_init_virtual: virtual ranks are replicas: same input width and noise key");
  TRY(ready(h, "dp_init_virtual", GAN));
  TRY(dp_switch(h, world, -1));
  h->dp_fused = true;
  dp_build_peers(h);
  return MRGAN_OK;
}

int mrgan_debug_buffer(mrgan_handle* h, int fold, int which, float* dst, int rows, int cols) {
  TRY(enter(h, "debug_buffer", FOLD, fold));
  if (!dst || rows < 1 || cols < 1) return fail(h, MRGAN_ERR_ARG, "debug_buffer: bad argument");
  TRY(ready(h, "debug_buffer", FOLD, fold));
  const FoldBuffers& b = h->fb[fold];
  const int K = h->cfg.n_classes, D = h->shapes[fold].D, nd = h->cfg.noise_dim;
  const bool gan = h->cfg.model == MRGAN_MODEL_GAN;
  const float* src = nullptr; int ld = 0;
  if (h->cfg.model == MRGAN_MODEL_SVM) {
    if (which != 50 && which != 51 && which != 60 && which != 61) return fail(h, MRGAN_ERR_STATE, "debug_buffer: an SVM handle has fold data and kernel matrices only");
    if (which >= 60) {
      if (!h->svm.fitted) return fail(h, MRGAN_ERR_STATE, "debug_buffer: kernel matrices before mrgan_svm_fit");
      if (rows > (which == 60 ? h->svm.n_lab : h->shapes[fold].n_test)) return fail(h, MRGAN_ERR_ARG, "debug_buffer: too many rows");
      src = which == 60 ? h->svm.Klab[fold] : h->svm.Kte[fold]; ld = h->svm.n_lab;
    }
  }
  if (which >= 0 && which <= 5) { src = b.a[which]; ld = b.lda[which]; }
  else if (which >= 11 && which <= 15) { src = b.hb[which - 10]; ld = b.lda[which - 10]; }
  else if (which >= 21 && which <= 25) { src = b.dz[which - 20]; ld = b.ldz[which - 20]; }
  else if (which == 30) { src = b.lg; ld = pitch8(K); }
  else if (which == 31) { src = b.dlg; ld = pitch8(K); }
  else if (which == 50) { src = b.xtr; ld = pitch8(D); }
  else if (which == 51) { src = b.xte; ld = b.lda[0]; }
  else if (gan && which == 32) { src = b.dfake; ld = pitch8(D); }
  else if (gan && which == 40) { src = b.zb; ld = pitch8(nd + 1); }
  else if (gan && which == 41) { src = b.h1g; ld = pitch8(kGH); }
  else if (gan && which == 42) { src = b.u; ld = pitch8(kGH + 1); }
  else if (gan && which == 43) { src = b.h2g; ld = pitch8(kGH + 1); }
  else if (gan && which == 44) { src = b.dz2g; ld = pitch8(kGH); }
  else if (gan && which == 45) { src = b.du; ld = pitch8(kGH); }
  else if (gan && which == 46) { src = b.dz1g; ld = pitch8(kGH); }
  if (!src || cols > ld) return fail(h, MRGAN_ERR_ARG, "debug_buffer: unknown buffer or too many columns");
  Temps tmp;
  if (h->om.mode == 2) {
    // f16 mode: noisy activations / inputs and every dZ exist only as fp16 operand copies (dZ times the loss scale)
    const bool act_only = (which >= 0 && which <= 4) || which == 40 || which == 42;
    const bool grad_only = (which >= 21 && which <= 25) || which == 31 || which == 32 || which == 44 || which == 46;
    float* t = nullptr;
    if (act_only || grad_only) {
      CK(tmp.alloc(&t, (size_t)rows * ld * sizeof(float)));
      launch_k(h, k_from_half, 256, 256, 0, h->stream, src, t, (size_t)rows * ld, grad_only ? 1.0f / h->om.gscale : 1.0f, h->om);
      src = t;
    } else if (which == 45) {   // du stays fp32 but carries the loss scale
      CK(tmp.alloc(&t, (size_t)rows * ld * sizeof(float)));
      CK(cudaMemcpyAsync(t, src, (size_t)rows * ld * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
      launch_k(h, k_scale_buf, 256, 256, 0, h->stream, t, (size_t)rows * ld, 1.0f / h->om.gscale);
      src = t;
    }
  }
  CK(cudaMemcpy2DAsync(dst, (size_t)cols * sizeof(float), src, (size_t)ld * sizeof(float), (size_t)cols * sizeof(float), rows,
                       cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

int mrgan_debug_gemm(mrgan_handle* h, int mode, int M, int N, int K, const float* A, const float* B, float* C, int use_tc) {
  TRY(enter(h, "debug_gemm", NETS));
  if (mode < 0 || mode > 2 || M < 1 || N < 1 || K < 1 || !A || !B || !C) return fail(h, MRGAN_ERR_ARG, "debug_gemm: bad argument");
  TRY(ready(h, "debug_gemm", NETS));
  // operand shapes (rows, cols) as stored
  const int ar = mode == 2 ? K : M, ac = mode == 2 ? M : K;
  const int br = mode == 1 ? N : K, bc = mode == 1 ? K : N;
  const int lda = pitch8(ac), ldb = pitch8(bc), ldc = pitch8(N);
  Temps tmp;
  float *dA = nullptr, *dB = nullptr, *dC = nullptr; GemmDesc* dd = nullptr;
  CK(tmp.alloc(&dA, (size_t)ar * lda * 4)); CK(tmp.alloc(&dB, (size_t)br * ldb * 4)); CK(tmp.alloc(&dC, (size_t)M * ldc * 4));
  CK(tmp.alloc(&dd, sizeof(GemmDesc)));
  CK(cudaMemsetAsync(dA, 0, (size_t)ar * lda * 4, h->stream)); CK(cudaMemsetAsync(dB, 0, (size_t)br * ldb * 4, h->stream));
  CK(cudaMemsetAsync(dC, 0, (size_t)M * ldc * 4, h->stream));
  CK(cudaMemcpy2DAsync(dA, (size_t)lda * 4, A, (size_t)ac * 4, (size_t)ac * 4, ar, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpy2DAsync(dB, (size_t)ldb * 4, B, (size_t)bc * 4, (size_t)bc * 4, br, cudaMemcpyHostToDevice, h->stream));
  GemmDesc g = make_desc(dA, lda, dB, ldb, dC, ldc, M, N, K, mode == 0 ? EPI_FWD : (mode == 1 ? EPI_DX : EPI_STORE), ACT_NONE, 0);
  CK(cudaMemcpyAsync(dd, &g, sizeof(g), cudaMemcpyHostToDevice, h->stream));
  if (use_tc == 2) {          // fp16 operand copies (kind::f16): host conversion, pitch rounded to 8 elements (16-byte TMA strides)
    const int lha = (ac + 7) & ~7, lhb = (bc + 7) & ~7;
    std::vector<__half> ha((size_t)ar * lha, __float2half(0.f)), hb((size_t)br * lhb, __float2half(0.f));
    for (int r = 0; r < ar; ++r) for (int c2 = 0; c2 < ac; ++c2) ha[(size_t)r * lha + c2] = __float2half_rn(A[(size_t)r * ac + c2]);
    for (int r = 0; r < br; ++r) for (int c2 = 0; c2 < bc; ++c2) hb[(size_t)r * lhb + c2] = __float2half_rn(B[(size_t)r * bc + c2]);
    __half *hA = nullptr, *hB = nullptr;
    CK(tmp.alloc(&hA, ha.size() * sizeof(__half))); CK(tmp.alloc(&hB, hb.size() * sizeof(__half)));
    CK(cudaMemcpy(hA, ha.data(), ha.size() * sizeof(__half), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(hB, hb.data(), hb.size() * sizeof(__half), cudaMemcpyHostToDevice));
    GemmDesc gh = g;
    gh.A = reinterpret_cast<const float*>(hA); gh.lda = lha; gh.B = reinterpret_cast<const float*>(hB); gh.ldb = lhb;
    TRY(tc_debug_gemm(h, mode, gh, 2));
  } else if (use_tc) {
    TRY(tc_debug_gemm(h, mode, g, 4));
  } else {
    const dim3 grid((N + 63) / 64, (M + 63) / 64, 1);
    if (mode == 0) launch_k(h, k_gemm_simt<false, false>, grid, 256, 0, h->stream, dd, h->d_folds, 0, h->hp);
    else if (mode == 1) launch_k(h, k_gemm_simt<false, true>, grid, 256, 0, h->stream, dd, h->d_folds, 0, h->hp);
    else launch_k(h, k_gemm_simt<true, false>, grid, 256, 0, h->stream, dd, h->d_folds, 0, h->hp);
  }
  CK(cudaMemcpy2DAsync(C, (size_t)N * 4, dC, (size_t)ldc * 4, (size_t)N * 4, M, cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

// ------------------------------------------------------------------ RBF C-SVC (MRGAN_MODEL_SVM, csrc/kernels_svm.cuh)
static void svm_launch(mrgan_handle* h, int phase) {
  mrgan_handle::Svm& S = h->svm;
  const int nf = h->nf;
  if (phase == MRGAN_TIME_SVM_KMAT) {
    launch_k(h, k_svm_split, dim3((S.max_rows + 7) / 8, 2 * nf), 256, 0, h->stream, S.d_split);
    launch_k(h, k_svm_kmat, dim3((S.n_lab + SVM_BM - 1) / SVM_BM, (S.max_rows + SVM_BN - 1) / SVM_BN, 2 * nf), SVM_KMAT_THREADS,
             SVM_KMAT_SMEM, h->stream, S.d_gemm);
  } else if (phase == MRGAN_TIME_SVM_SMO) {
    launch_k(h, k_svm_smo, nf * S.npairs, SVM_SMO_THREADS, (size_t)SVM_SMO_SMEM_PER_ROW * S.npmax, h->stream, S.d_jobs, S.eps);
  } else {
    launch_k(h, k_svm_vote, dim3(S.max_nte, nf), SVM_VOTE_THREADS, 0, h->stream, S.d_jobs, S.npairs, h->cfg.n_classes, S.d_Kt, nullptr,
             S.d_yte, S.d_nte, S.d_dec, S.d_wrong, S.d_pred);
    launch_k(h, k_svm_count, nf, 256, 0, h->stream, S.d_wrong, S.d_nte, S.d_count);
  }
}

// The labeled rows of every fold: class c is the segment [start[f][c], start[f][c] + cnt[f][c]); ylab [nf][n_lab] their labels
struct SvmLabels {
  std::vector<int> ylab, start, cnt;
  int npmax = 0;                      // rows of the largest class pair
};

// Checks the labeled rows of every loaded fold (in range, class-major, every class present, class pairs within SVM_MAX_PAIR)
// and reads their labels.  Changes no SVM state.  The caller has checked the scalars.
static int svm_labels(mrgan_handle* h, const char* fn, const int32_t* lab_rows, int n_lab, SvmLabels& L) {
  const std::string pre = std::string(fn) + ": ";
  const int nf = h->nf, K = h->cfg.n_classes;
  std::vector<int> ytr(h->n_train);
  std::vector<int>& ylab = L.ylab;
  std::vector<int>& start = L.start;
  std::vector<int>& cnt = L.cnt;
  ylab.assign((size_t)nf * n_lab, 0);
  start.assign((size_t)nf * K, 0);
  cnt.assign((size_t)nf * K, 0);
  int& npmax = L.npmax;
  npmax = 0;
  for (int f = 0; f < nf; ++f) {
    CK(cudaMemcpy(ytr.data(), h->fb[f].ytr, (size_t)h->n_train * sizeof(int), cudaMemcpyDeviceToHost));
    const int32_t* lr = lab_rows + (size_t)f * n_lab;
    int prev = -1;
    for (int r = 0; r < n_lab; ++r) {
      if (lr[r] < 0 || lr[r] >= h->n_train) return fail(h, MRGAN_ERR_ARG, pre + "labeled row out of range");
      const int c = ytr[lr[r]];
      if (c < prev) return fail(h, MRGAN_ERR_ARG, pre + "labeled rows must be class-major (labels non-decreasing)");
      if (c != prev) start[(size_t)f * K + c] = r;
      cnt[(size_t)f * K + c]++;
      ylab[(size_t)f * n_lab + r] = c;
      prev = c;
    }
    for (int c = 0; c < K; ++c)
      if (cnt[(size_t)f * K + c] == 0) return fail(h, MRGAN_ERR_ARG, pre + "every class needs a labeled row");
    for (int a = 0; a < K; ++a)
      for (int b = a + 1; b < K; ++b) {
        const int np = cnt[(size_t)f * K + a] + cnt[(size_t)f * K + b];
        if (np > SVM_MAX_PAIR) return fail(h, MRGAN_ERR_ARG, pre + "a class pair has more than 8192 labeled rows (shared-memory limit of the solver)");
        npmax = std::max(npmax, np);
      }
  }
  return MRGAN_OK;
}

// Lays out the fit's workspace for checked labeled rows and uploads its descriptors: the operand split and both kernel
// matrices of every fold at gamma[f], and one problem per (fold, class pair) at C[f] over the fold's contiguous class
// segments.  Launches nothing; the previous fit is invalid from here on.
static int svm_setup(mrgan_handle* h, const int32_t* lab_rows, int n_lab, const SvmLabels& L, const float* C, const float* gamma,
                     float tol) {
  const int nf = h->nf, K = h->cfg.n_classes, npairs = K * (K - 1) / 2, npmax = L.npmax;
  const std::vector<int>& start = L.start;
  const std::vector<int>& cnt = L.cnt;
  mrgan_handle::Svm& S = h->svm;
  int max_nte = 0, max_kp = 32;
  for (int f = 0; f < nf; ++f) { max_nte = std::max(max_nte, h->shapes[f].n_test); max_kp = std::max(max_kp, round_up(h->shapes[f].D, 32)); }
  std::vector<float*> Hl(nf), Ll(nf), Ht(nf), Lt(nf), Klab(nf), Kte(nf), dec(nf);
  std::vector<double*> nl(nf), nt(nf), coef(nf), rho(nf);
  std::vector<int*> wrong(nf);
  int* d_lab = nullptr;
  auto layout = [&](Arena& ar) {
    for (int f = 0; f < nf; ++f) {
      const int Kp = round_up(h->shapes[f].D, 32), nte = h->shapes[f].n_test;
      Hl[f] = ar.take<float>((size_t)n_lab * Kp); Ll[f] = ar.take<float>((size_t)n_lab * Kp);
      Ht[f] = ar.take<float>((size_t)nte * Kp); Lt[f] = ar.take<float>((size_t)nte * Kp);
      nl[f] = ar.take<double>(n_lab); nt[f] = ar.take<double>(nte);
      Klab[f] = ar.take<float>((size_t)n_lab * n_lab); Kte[f] = ar.take<float>((size_t)nte * n_lab);
      coef[f] = ar.take<double>((size_t)npairs * npmax); rho[f] = ar.take<double>(npairs);
      dec[f] = ar.take<float>((size_t)nte * npairs); wrong[f] = ar.take<int>(nte);
    }
    d_lab = ar.take<int>((size_t)nf * n_lab);
    S.d_iters = ar.take<int>((size_t)nf * npairs); S.d_capped = ar.take<int>((size_t)nf * npairs);
    S.d_count = ar.take<int>(nf); S.d_nte = ar.take<int>(nf);
    S.d_split = ar.take<SvmSplitOp>(2 * nf); S.d_gemm = ar.take<SvmGemmOp>(2 * nf); S.d_jobs = ar.take<SvmPairJob>((size_t)nf * npairs);
    S.d_Kt = ar.take<float*>(nf); S.d_dec = ar.take<float*>(nf); S.d_yte = ar.take<int*>(nf); S.d_wrong = ar.take<int*>(nf);
    S.d_pred = ar.take<int*>(nf);
    S.Xs = ar.take<float>((size_t)max_nte * max_kp); S.Hs = ar.take<float>((size_t)max_nte * max_kp); S.Ls = ar.take<float>((size_t)max_nte * max_kp);
    S.ns = ar.take<double>(max_nte); S.Ks = ar.take<float>((size_t)max_nte * n_lab); S.decs = ar.take<float>((size_t)max_nte * npairs);
    S.preds = ar.take<int>(max_nte);
    S.d_split_s = ar.take<SvmSplitOp>(1); S.d_gemm_s = ar.take<SvmGemmOp>(1);
    S.d_Ks = ar.take<float*>(1); S.d_decs = ar.take<float*>(1); S.d_preds = ar.take<int*>(1); S.d_ns = ar.take<int>(1);
  };
  Arena sizing;
  layout(sizing);
  S.fitted = false;
  if (sizing.off + 256 > S.bytes) {
    if (S.mem) { cudaFree(S.mem); S.mem = nullptr; S.bytes = 0; }
    CK(cudaMalloc(&S.mem, sizing.off + 256));
    S.bytes = sizing.off + 256;
  }
  Arena real; real.base = S.mem;
  layout(real);
  S.n_lab = n_lab; S.npairs = npairs; S.npmax = npmax; S.max_nte = max_nte; S.max_rows = std::max(n_lab, max_nte);
  S.eps = tol;
  S.Klab = Klab; S.Kte = Kte; S.dec = dec; S.wrong = wrong;
  // descriptors
  EncodeTiledFn enc = tc_encoder();
  if (!enc) return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  std::vector<SvmSplitOp> sp(2 * nf);
  std::vector<SvmGemmOp> gm(2 * nf);
  std::vector<SvmPairJob> jobs((size_t)nf * npairs);
  std::vector<int> nte_v(nf);
  std::vector<int*> yte_v(nf), pred_v(nf);
  memset(gm.data(), 0, sizeof(SvmGemmOp) * gm.size());
  for (int f = 0; f < nf; ++f) {
    const FoldBuffers& b = h->fb[f];
    const int D = h->shapes[f].D, Kp = round_up(D, 32), nte = h->shapes[f].n_test;
    sp[2 * f] = SvmSplitOp{b.xtr, pitch8(D), d_lab + (size_t)f * n_lab, n_lab, D, Kp, Hl[f], Ll[f], nl[f]};
    sp[2 * f + 1] = SvmSplitOp{b.xte, b.lda[0], nullptr, nte, D, Kp, Ht[f], Lt[f], nt[f]};
    for (int w = 0; w < 2; ++w) {
      SvmGemmOp& g = gm[2 * f + w];
      const int nA = w == 0 ? n_lab : nte;
      bool ok = make_map(enc, &g.mapBh, Hl[f], Kp, n_lab, Kp, SVM_BM, false) && make_map(enc, &g.mapBl, Ll[f], Kp, n_lab, Kp, SVM_BM, false) &&
                make_map(enc, &g.mapAh, w == 0 ? Hl[f] : Ht[f], Kp, nA, Kp, SVM_BN, false) &&
                make_map(enc, &g.mapAl, w == 0 ? Ll[f] : Lt[f], Kp, nA, Kp, SVM_BN, false);
      if (!ok) return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled failed");
      g.normA = w == 0 ? nl[f] : nt[f]; g.normB = nl[f];
      g.C = w == 0 ? Klab[f] : Kte[f]; g.ldc = n_lab;
      g.nA = nA; g.nB = n_lab; g.Kp = Kp; g.gamma = gamma[f]; g.same = w == 0;
    }
    int p = 0;
    for (int a = 0; a < K; ++a)
      for (int c = a + 1; c < K; ++c, ++p) {
        SvmPairJob& jb = jobs[(size_t)f * npairs + p];
        jb.K = Klab[f]; jb.ld = n_lab;
        jb.a_off = start[(size_t)f * K + a]; jb.na = cnt[(size_t)f * K + a];
        jb.b_off = start[(size_t)f * K + c]; jb.nb = cnt[(size_t)f * K + c];
        jb.rows = nullptr; jb.C = C[f];
        jb.ca = a; jb.cb = c;
        jb.coef = coef[f] + (size_t)p * npmax; jb.rho = rho[f] + p;
        jb.n_iter = S.d_iters + (size_t)f * npairs + p; jb.capped = S.d_capped + (size_t)f * npairs + p;
      }
    nte_v[f] = nte; yte_v[f] = b.yte; pred_v[f] = b.pred;
  }
  S.h_gemm = gm;
  CK(cudaMemcpyAsync(d_lab, lab_rows, (size_t)nf * n_lab * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_split, sp.data(), sizeof(SvmSplitOp) * sp.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_gemm, gm.data(), sizeof(SvmGemmOp) * gm.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_jobs, jobs.data(), sizeof(SvmPairJob) * jobs.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_nte, nte_v.data(), sizeof(int) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_Kt, Kte.data(), sizeof(float*) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_dec, dec.data(), sizeof(float*) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_yte, yte_v.data(), sizeof(int*) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_wrong, wrong.data(), sizeof(int*) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_pred, pred_v.data(), sizeof(int*) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_Ks, &S.Ks, sizeof(float*), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_decs, &S.decs, sizeof(float*), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.d_preds, &S.preds, sizeof(int*), cudaMemcpyHostToDevice, h->stream));
  CK(cudaFuncSetAttribute(k_svm_kmat, cudaFuncAttributeMaxDynamicSharedMemorySize, SVM_KMAT_SMEM));
  CK(cudaFuncSetAttribute(k_svm_smo, cudaFuncAttributeMaxDynamicSharedMemorySize, SVM_SMO_SMEM_PER_ROW * SVM_MAX_PAIR));
  return MRGAN_OK;
}

static bool all_positive(const float* v, size_t n) {
  for (size_t i = 0; i < n; ++i)
    if (!(v[i] > 0.0f)) return false;
  return true;
}

int mrgan_svm_fit_folds(mrgan_handle* h, const int32_t* lab_rows, int n_lab, const float* C, const float* gamma, float tol, int32_t* n_iter) {
  TRY(enter(h, "svm_fit", SVM));
  if (!lab_rows || !C || !gamma || n_lab < 2 || !(tol > 0.0f)) return fail(h, MRGAN_ERR_ARG, "svm_fit: bad argument");
  const int nf = h->nf, npairs = h->cfg.n_classes * (h->cfg.n_classes - 1) / 2;
  if (!all_positive(C, nf)) return fail(h, MRGAN_ERR_ARG, "svm_fit: C must be positive");
  if (!all_positive(gamma, nf)) return fail(h, MRGAN_ERR_ARG, "svm_fit: gamma must be positive");
  TRY(ready(h, "svm_fit", SVM | LOADED));
  SvmLabels L;
  TRY(svm_labels(h, "svm_fit", lab_rows, n_lab, L));
  TRY(svm_setup(h, lab_rows, n_lab, L, C, gamma, tol));
  mrgan_handle::Svm& S = h->svm;
  svm_launch(h, MRGAN_TIME_SVM_KMAT);
  svm_launch(h, MRGAN_TIME_SVM_SMO);
  svm_launch(h, MRGAN_TIME_SVM_PREDICT);
  std::vector<int> it((size_t)nf * npairs), cap((size_t)nf * npairs);
  CK(cudaMemcpyAsync(it.data(), S.d_iters, sizeof(int) * it.size(), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(cap.data(), S.d_capped, sizeof(int) * cap.size(), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  if (n_iter) memcpy(n_iter, it.data(), sizeof(int) * it.size());
  S.fitted = true;
  for (size_t q = 0; q < cap.size(); ++q)
    if (cap[q]) return fail(h, MRGAN_ERR_STATE, "svm_fit: fold " + std::to_string(q / npairs) + ", class pair " + std::to_string(q % npairs) +
                                                    " hit the iteration cap max(1e7, 100 n)");
  return MRGAN_OK;
}

int mrgan_svm_fit(mrgan_handle* h, const int32_t* lab_rows, int n_lab, float C, const float* gamma, float tol, int32_t* n_iter) {
  TRY(enter(h, "svm_fit", 0));
  std::vector<float> Cf(h->nf, C);
  return mrgan_svm_fit_folds(h, lab_rows, n_lab, Cf.data(), gamma, tol, n_iter);
}

// Inner cross-validation (GridSearchCV's fits and scores): for every gamma column g, the labeled x labeled kernel matrices
// of all folds are recomputed in the fit's buffers, then one SMO problem per (fold, C, split, class pair) is solved on the
// split's inner-training rows (a row map into the labeled set) and the split's validation rows are voted from the same
// matrix and counted.
int mrgan_svm_cv(mrgan_handle* h, const int32_t* lab_rows, int n_lab, const int32_t* split, int n_splits, const float* C, int nC,
                 const float* gamma, int nG, float tol, int32_t* wrong) {
  TRY(enter(h, "svm_cv", SVM));
  if (!lab_rows || !split || !C || !gamma || !wrong || n_lab < 2 || !(tol > 0.0f)) return fail(h, MRGAN_ERR_ARG, "svm_cv: bad argument");
  if (n_splits < 2 || nC < 1 || nG < 1) return fail(h, MRGAN_ERR_ARG, "svm_cv: need n_splits >= 2, nC >= 1 and nG >= 1");
  const int nf = h->nf, K = h->cfg.n_classes, npairs = K * (K - 1) / 2, ns = n_splits;
  if (!all_positive(C, nC)) return fail(h, MRGAN_ERR_ARG, "svm_cv: C must be positive");
  if (!all_positive(gamma, (size_t)nf * nG)) return fail(h, MRGAN_ERR_ARG, "svm_cv: gamma must be positive");
  for (size_t r = 0; r < (size_t)nf * n_lab; ++r)
    if (split[r] < 0 || split[r] >= ns) return fail(h, MRGAN_ERR_ARG, "svm_cv: split index outside [0, n_splits)");
  std::vector<float> g0(nf), C0(nf, C[0]);
  for (int f = 0; f < nf; ++f) g0[f] = gamma[(size_t)f * nG];
  TRY(ready(h, "svm_cv", SVM | LOADED));
  SvmLabels L;
  TRY(svm_labels(h, "svm_cv", lab_rows, n_lab, L));
  const std::vector<int>& ylab = L.ylab;
  // the problems: validation rows of (f, s) and the inner-training rows of (f, s, pair), in the labeled order; a rejected
  // split leaves the previous fit valid
  const int nQ = nf * nC * ns, nJobs = nQ * npairs;
  std::vector<int> vrows, vy, voff((size_t)nf * ns), nval((size_t)nf * ns, 0), maps, moff((size_t)nf * ns * npairs), mna(moff.size()), mnb(moff.size());
  int max_nval = 0, npmax = 0;
  for (int f = 0; f < nf; ++f) {
    const int32_t* sf = split + (size_t)f * n_lab;
    const int* yf = ylab.data() + (size_t)f * n_lab;
    for (int s = 0; s < ns; ++s) {
      const size_t fs = (size_t)f * ns + s;
      voff[fs] = (int)vrows.size();
      std::vector<int> train_cnt(K, 0);
      for (int r = 0; r < n_lab; ++r) {
        if (sf[r] == s) { vrows.push_back(r); vy.push_back(yf[r]); }
        else train_cnt[yf[r]]++;
      }
      nval[fs] = (int)vrows.size() - voff[fs];
      if (nval[fs] == 0) return fail(h, MRGAN_ERR_ARG, "svm_cv: fold " + std::to_string(f) + ", split " + std::to_string(s) + " has no validation row");
      for (int c = 0; c < K; ++c)
        if (train_cnt[c] == 0)
          return fail(h, MRGAN_ERR_ARG, "svm_cv: fold " + std::to_string(f) + ", split " + std::to_string(s) + ": the inner-training rows lack class " + std::to_string(c));
      max_nval = std::max(max_nval, nval[fs]);
      int p = 0;
      for (int a = 0; a < K; ++a)
        for (int b = a + 1; b < K; ++b, ++p) {
          const size_t m = fs * npairs + p;
          moff[m] = (int)maps.size();
          for (int r = 0; r < n_lab; ++r) if (sf[r] != s && yf[r] == a) maps.push_back(r);
          mna[m] = (int)maps.size() - moff[m];
          for (int r = 0; r < n_lab; ++r) if (sf[r] != s && yf[r] == b) maps.push_back(r);
          mnb[m] = (int)maps.size() - moff[m] - mna[m];
          npmax = std::max(npmax, mna[m] + mnb[m]);
        }
    }
  }
  TRY(svm_setup(h, lab_rows, n_lab, L, C0.data(), g0.data(), tol));
  mrgan_handle::Svm& S = h->svm;
  // second allocation: kept while large enough, freed by mrgan_destroy
  int *d_maps = nullptr, *d_vrows = nullptr, *d_vy = nullptr, *d_nval = nullptr, *d_flags = nullptr, *d_count = nullptr, *d_iters = nullptr, *d_capped = nullptr;
  double *d_coef = nullptr, *d_rho = nullptr;
  SvmPairJob* d_jobs = nullptr; SvmGemmOp* d_gemm = nullptr;
  const float** d_Kq = nullptr; const int** d_trow = nullptr; const int** d_yq = nullptr; int** d_wq = nullptr;
  auto layout = [&](Arena& ar) {
    d_maps = ar.take<int>(maps.size()); d_vrows = ar.take<int>(vrows.size()); d_vy = ar.take<int>(vy.size());
    d_nval = ar.take<int>(nQ); d_flags = ar.take<int>((size_t)nQ * max_nval); d_count = ar.take<int>((size_t)nG * nQ);
    d_iters = ar.take<int>(nJobs); d_capped = ar.take<int>(nJobs);
    d_coef = ar.take<double>((size_t)nJobs * npmax); d_rho = ar.take<double>(nJobs);
    d_jobs = ar.take<SvmPairJob>(nJobs); d_gemm = ar.take<SvmGemmOp>((size_t)nG * nf);
    d_Kq = ar.take<const float*>(nQ); d_trow = ar.take<const int*>(nQ); d_yq = ar.take<const int*>(nQ); d_wq = ar.take<int*>(nQ);
  };
  Arena sizing;
  layout(sizing);
  if (sizing.off + 256 > S.cv_bytes) {
    if (S.cv_mem) { cudaFree(S.cv_mem); S.cv_mem = nullptr; S.cv_bytes = 0; }
    CK(cudaMalloc(&S.cv_mem, sizing.off + 256));
    S.cv_bytes = sizing.off + 256;
  }
  Arena real; real.base = S.cv_mem;
  layout(real);
  // problem q = (f * nC + c) * ns + s; its class pairs are jobs q * npairs ...
  std::vector<SvmPairJob> jobs(nJobs);
  std::vector<const float*> Kq(nQ); std::vector<const int*> trow(nQ), yq(nQ); std::vector<int*> wq(nQ); std::vector<int> nq(nQ);
  for (int f = 0; f < nf; ++f)
    for (int c = 0; c < nC; ++c)
      for (int s = 0; s < ns; ++s) {
        const int q = (f * nC + c) * ns + s;
        const size_t fs = (size_t)f * ns + s;
        Kq[q] = S.Klab[f]; trow[q] = d_vrows + voff[fs]; yq[q] = d_vy + voff[fs]; wq[q] = d_flags + (size_t)q * max_nval; nq[q] = nval[fs];
        int p = 0;
        for (int a = 0; a < K; ++a)
          for (int b = a + 1; b < K; ++b, ++p) {
            const size_t m = fs * npairs + p, j = (size_t)q * npairs + p;
            SvmPairJob& jb = jobs[j];
            jb.K = S.Klab[f]; jb.ld = n_lab;
            jb.rows = d_maps + moff[m]; jb.na = mna[m]; jb.nb = mnb[m];
            jb.C = C[c]; jb.ca = a; jb.cb = b;
            jb.coef = d_coef + j * npmax; jb.rho = d_rho + j;
            jb.n_iter = d_iters + j; jb.capped = d_capped + j;
          }
      }
  std::vector<SvmGemmOp> gm((size_t)nG * nf);
  for (int g = 0; g < nG; ++g)
    for (int f = 0; f < nf; ++f) {
      gm[(size_t)g * nf + f] = S.h_gemm[2 * f];
      gm[(size_t)g * nf + f].gamma = gamma[(size_t)f * nG + g];
    }
  CK(cudaMemcpyAsync(d_maps, maps.data(), sizeof(int) * maps.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_vrows, vrows.data(), sizeof(int) * vrows.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_vy, vy.data(), sizeof(int) * vy.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_nval, nq.data(), sizeof(int) * nQ, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(SvmPairJob) * jobs.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_gemm, gm.data(), sizeof(SvmGemmOp) * gm.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_Kq, Kq.data(), sizeof(float*) * nQ, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_trow, trow.data(), sizeof(int*) * nQ, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_yq, yq.data(), sizeof(int*) * nQ, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_wq, wq.data(), sizeof(int*) * nQ, cudaMemcpyHostToDevice, h->stream));
  // the operand split does not depend on gamma: once (the fit's launch, which also splits the test rows)
  launch_k(h, k_svm_split, dim3((S.max_rows + 7) / 8, 2 * nf), 256, 0, h->stream, S.d_split);
  std::vector<int> cap(nJobs), cnt((size_t)nG * nQ);
  for (int g = 0; g < nG; ++g) {
    launch_k(h, k_svm_kmat, dim3((n_lab + SVM_BM - 1) / SVM_BM, (n_lab + SVM_BN - 1) / SVM_BN, nf), SVM_KMAT_THREADS, SVM_KMAT_SMEM,
             h->stream, d_gemm + (size_t)g * nf);
    launch_k(h, k_svm_smo, nJobs, SVM_SMO_THREADS, (size_t)SVM_SMO_SMEM_PER_ROW * npmax, h->stream, d_jobs, S.eps);
    launch_k(h, k_svm_vote, dim3(max_nval, nQ), SVM_VOTE_THREADS, 0, h->stream, d_jobs, npairs, K, d_Kq, d_trow, d_yq, d_nval, nullptr,
             d_wq, nullptr);
    launch_k(h, k_svm_count, nQ, 256, 0, h->stream, d_wq, d_nval, d_count + (size_t)g * nQ);
    CK(cudaMemcpyAsync(cap.data(), d_capped, sizeof(int) * nJobs, cudaMemcpyDeviceToHost, h->stream));
    TRY(complete(h));
    for (int j = 0; j < nJobs; ++j)
      if (cap[j]) {
        const int q = j / npairs, s = q % ns, c = (q / ns) % nC, f = q / (ns * nC);
        return fail(h, MRGAN_ERR_STATE, "svm_cv: fold " + std::to_string(f) + ", gamma " + std::to_string(g) + ", C " + std::to_string(c) +
                                         ", split " + std::to_string(s) + ", class pair " + std::to_string(j % npairs) +
                                         " hit the iteration cap max(1e7, 100 n)");
      }
  }
  CK(cudaMemcpyAsync(cnt.data(), d_count, sizeof(int) * cnt.size(), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  for (int f = 0; f < nf; ++f)
    for (int g = 0; g < nG; ++g)
      for (int c = 0; c < nC; ++c)
        for (int s = 0; s < ns; ++s) wrong[(((size_t)f * nG + g) * nC + c) * ns + s] = cnt[(size_t)g * nQ + (f * nC + c) * ns + s];
  return MRGAN_OK;
}

int mrgan_svm_eval(mrgan_handle* h, int fold, float* err) {
  TRY(enter(h, "svm_eval", FOLD | SVM, fold));
  if (!err) return fail(h, MRGAN_ERR_ARG, "svm_eval: null pointer");
  TRY(ready(h, "svm_eval", FOLD | SVM | FITTED, fold));
  int c = 0;
  CK(cudaMemcpyAsync(&c, h->svm.d_count + fold, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  *err = (float)c / (float)h->shapes[fold].n_test;     // np.mean(predicted != y_test)
  return MRGAN_OK;
}

int mrgan_svm_decision(mrgan_handle* h, int fold, float* dst) {
  TRY(enter(h, "svm_decision", FOLD | SVM, fold));
  if (!dst) return fail(h, MRGAN_ERR_ARG, "svm_decision: null pointer");
  TRY(ready(h, "svm_decision", FOLD | SVM | FITTED, fold));
  CK(cudaMemcpyAsync(dst, h->svm.dec[fold], sizeof(float) * h->shapes[fold].n_test * h->svm.npairs, cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

// ------------------------------------------------------------------ predictions and confusion counts
int mrgan_predict(mrgan_handle* h, int fold, int32_t* pred, float* scores) {
  TRY(enter(h, "predict", FOLD, fold));
  if (!pred) return fail(h, MRGAN_ERR_ARG, "predict: null pointer");
  const bool svm = h->cfg.model == MRGAN_MODEL_SVM;
  TRY(ready(h, "predict", FOLD | LOCAL | (svm ? FITTED : LOADED), fold));
  const int n = h->shapes[fold].n_test, K = h->cfg.n_classes;
  const FoldBuffers& b = h->fb[fold];
  if (svm) {
    CK(cudaMemcpyAsync(pred, b.pred, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));     // voted by mrgan_svm_fit
    if (scores) CK(cudaMemcpyAsync(scores, h->svm.dec[fold], (size_t)n * h->svm.npairs * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  } else {
    enqueue_eval(h, fold, 1, false, 0, true);
    CK(cudaMemcpyAsync(pred, b.pred, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (scores)
      CK(cudaMemcpy2DAsync(scores, (size_t)K * sizeof(float), b.elg, (size_t)pitch8(K) * sizeof(float), (size_t)K * sizeof(float), n,
                           cudaMemcpyDeviceToHost, h->stream));
  }
  return complete(h);
}

int mrgan_predict_rows(mrgan_handle* h, int fold, const float* x, int n, int32_t* pred, float* scores) {
  TRY(enter(h, "predict_rows", FOLD, fold));
  if (!x || !pred) return fail(h, MRGAN_ERR_ARG, "predict_rows: null pointer");
  if (n < 1 || n > h->shapes[fold].n_test) return fail(h, MRGAN_ERR_ARG, "predict_rows: n must be in [1, n_test of the fold]");
  const bool svm = h->cfg.model == MRGAN_MODEL_SVM;
  TRY(ready(h, "predict_rows", FOLD | LOCAL | (svm ? FITTED : LOADED), fold));
  const int D = h->shapes[fold].D, K = h->cfg.n_classes;
  FoldBuffers& b = h->fb[fold];
  if (svm) {
    mrgan_handle::Svm& S = h->svm;
    EncodeTiledFn fn = tc_encoder();
    if (!fn) return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    // the new rows replace the fold's test rows in its second kernel-matrix descriptor (labeled rows, norms, gamma kept)
    const int Kp = round_up(D, 32);
    SvmSplitOp sp{S.Xs, Kp, nullptr, n, D, Kp, S.Hs, S.Ls, S.ns};
    SvmGemmOp g = S.h_gemm[2 * fold + 1];
    if (!make_map(fn, &g.mapAh, S.Hs, Kp, n, Kp, SVM_BN, false) || !make_map(fn, &g.mapAl, S.Ls, Kp, n, Kp, SVM_BN, false))
      return fail(h, MRGAN_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    g.normA = S.ns; g.C = S.Ks; g.nA = n;
    const size_t w = (size_t)D * sizeof(float);
    CK(cudaMemcpy2DAsync(S.Xs, (size_t)Kp * sizeof(float), x, w, w, n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(S.d_split_s, &sp, sizeof(sp), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(S.d_gemm_s, &g, sizeof(g), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(S.d_ns, &n, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    launch_k(h, k_svm_split, dim3((n + 7) / 8, 1), 256, 0, h->stream, S.d_split_s);
    launch_k(h, k_svm_kmat, dim3((S.n_lab + SVM_BM - 1) / SVM_BM, (n + SVM_BN - 1) / SVM_BN, 1), SVM_KMAT_THREADS, SVM_KMAT_SMEM, h->stream,
             S.d_gemm_s);
    launch_k(h, k_svm_vote, dim3(n, 1), SVM_VOTE_THREADS, 0, h->stream, S.d_jobs + (size_t)fold * S.npairs, S.npairs, K, S.d_Ks, nullptr,
             nullptr, S.d_ns, S.d_decs, nullptr, S.d_preds);
    CK(cudaMemcpyAsync(pred, S.preds, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (scores) CK(cudaMemcpyAsync(scores, S.decs, (size_t)n * S.npairs * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  } else {
    // the staging path of mrgan_test_batch, without labels (the error it computes on the stale staged labels is unused)
    TRY(stage_rows(h, fold, x, n));
    enqueue_eval(h, fold, 1, true, n, true);
    CK(cudaMemcpyAsync(pred, b.pred_s, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (scores)
      CK(cudaMemcpy2DAsync(scores, (size_t)K * sizeof(float), b.elg, (size_t)pitch8(K) * sizeof(float), (size_t)K * sizeof(float), n,
                           cudaMemcpyDeviceToHost, h->stream));
  }
  return complete(h);
}

int mrgan_confusion(mrgan_handle* h, int32_t* out) {
  TRY(enter(h, "confusion", 0));
  if (!out) return fail(h, MRGAN_ERR_ARG, "confusion: null pointer");
  const bool svm = h->cfg.model == MRGAN_MODEL_SVM;
  TRY(ready(h, "confusion", LOCAL | (svm ? FITTED : LOADED)));
  const int K = h->cfg.n_classes;
  if (!svm) enqueue_eval(h, 0, h->nf, false, 0, true);   // every fold in one pass; the SVM voted at fit
  enqueue_confusion(h);
  CK(cudaMemcpyAsync(out, h->d_conf, (size_t)h->nf * K * K * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

// ------------------------------------------------------------------ input gradients and saliency profiles
int mrgan_input_grad(mrgan_handle* h, int fold, const float* x, int n, const int32_t* target, float* grad) {
  TRY(enter(h, "input_grad", FOLD | NETS, fold));
  if (!grad) return fail(h, MRGAN_ERR_ARG, "input_grad: null pointer");
  const int D = h->shapes[fold].D, K = h->cfg.n_classes, nte = h->shapes[fold].n_test;
  if (n < 1 || n > nte) return fail(h, MRGAN_ERR_ARG, "input_grad: n must be in [1, n_test of the fold]");
  if (!x && n != nte) return fail(h, MRGAN_ERR_ARG, "input_grad: the resident test set (x = NULL) has n_test rows");
  if (target)
    for (int i = 0; i < n; ++i)
      if (target[i] < 0 || target[i] >= K) return fail(h, MRGAN_ERR_ARG, "input_grad: target class out of range");
  TRY(ready(h, "input_grad", FOLD | NETS | LOCAL | LOADED, fold));
  TRY(saliency_setup(h));
  FoldBuffers& b = h->fb[fold];
  const size_t w = (size_t)D * sizeof(float), ld0 = (size_t)b.lda[0] * sizeof(float);
  if (x) TRY(stage_rows(h, fold, x, n));
  if (target) CK(cudaMemcpyAsync(b.ey_stage, target, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  enqueue_input_grad(h, fold, 1, x != nullptr, x ? n : 0, target ? TGT_STAGED : TGT_PRED);
  CK(cudaMemcpy2DAsync(grad, w, b.ex_stage, ld0, w, n, cudaMemcpyDeviceToHost, h->stream));
  return complete(h);
}

int mrgan_saliency(mrgan_handle* h, float* profile) {
  TRY(enter(h, "saliency", NETS));
  if (!profile) return fail(h, MRGAN_ERR_ARG, "saliency: null pointer");
  TRY(ready(h, "saliency", NETS | LOCAL | LOADED));
  TRY(saliency_setup(h));
  enqueue_saliency(h);
  CK(cudaMemcpyAsync(profile, h->sal.profile, (size_t)h->nf * h->cfg.n_classes * max_D(h, 0, h->nf) * sizeof(float), cudaMemcpyDeviceToHost,
                     h->stream));
  return complete(h);
}

// ------------------------------------------------------------------ samples of the generator (include/mrgan.h)
int mrgan_generate(mrgan_handle* h, int fold, int n, uint32_t seed, const float* z, float* x) {
  TRY(enter(h, "generate", FOLD | GAN, fold));
  if (!x) return fail(h, MRGAN_ERR_ARG, "generate: null pointer");
  if (n < 1 || n % h->cfg.batch) return fail(h, MRGAN_ERR_ARG, "generate: n must be a positive multiple of batch");
  TRY(ready(h, "generate", FOLD | GAN | LOCAL, fold));
  TRY(gen_setup(h));
  const mrgan_handle::GenWork& G = h->gen;
  const int D = h->shapes[fold].D, nd = h->cfg.noise_dim;
  const GemmDesc& g3 = h->h_descs[(size_t)OP_GG3 * h->nf + fold];     // C: the clean rows
  for (int r0 = 0; r0 < n; r0 += G.NG) {
    const int c = std::min(G.NG, n - r0);
    if (z) CK(cudaMemcpyAsync(G.zs, z + (size_t)r0 * nd, (size_t)c * nd * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    enqueue_generate(h, fold, 1, r0, c, seed, z != nullptr);
    CK(cudaMemcpy2DAsync(x + (size_t)r0 * D, (size_t)D * sizeof(float), g3.C, (size_t)g3.ldc * sizeof(float), (size_t)D * sizeof(float), c,
                         cudaMemcpyDeviceToHost, h->stream));
  }
  return complete(h);
}

int mrgan_sample_stats(mrgan_handle* h, int n, uint32_t seed, int32_t* counts, double* score, double* mean, double* cov) {
  TRY(enter(h, "sample_stats", GAN));
  if (!counts || !score || !mean || !cov) return fail(h, MRGAN_ERR_ARG, "sample_stats: null pointer");
  if (n < 1 || n % h->cfg.batch) return fail(h, MRGAN_ERR_ARG, "sample_stats: n must be a positive multiple of batch");
  TRY(ready(h, "sample_stats", GAN | LOCAL | LOADED));
  TRY(gen_setup(h));
  const mrgan_handle::GenWork& G = h->gen;
  const int nf = h->nf, K = h->cfg.n_classes, W = SS_W;
  enqueue_sample_stats(h, n, seed);
  std::vector<double> s1((size_t)nf * 2 * W), s2((size_t)nf * 2 * W * W), sc((size_t)nf * 2);
  std::vector<int> cnt((size_t)nf * 64);
  CK(cudaMemcpyAsync(s1.data(), G.s1, s1.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(s2.data(), G.s2, s2.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(sc.data(), G.score, sc.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(cnt.data(), G.counts, cnt.size() * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  TRY(complete(h));
  // raw sums -> moments: mean = s1 / m, cov = (s2 - m mean mean^T) / (m - 1) (np.cov), s2 mirrored from its upper triangle
  for (int f = 0; f < nf; ++f) {
    for (int k = 0; k < K; ++k) counts[(size_t)f * K + k] = cnt[(size_t)f * 64 + k];
    for (int side = 0; side < 2; ++side) {
      const double m = side ? h->shapes[f].n_test : n;
      const size_t fs = (size_t)f * 2 + side;
      const double* a = s1.data() + fs * W;
      const double* q = s2.data() + fs * W * W;
      double* mu = mean + fs * W;
      double* cv = cov + fs * W * W;
      score[fs] = sc[fs] / m;
      for (int i = 0; i < W; ++i) mu[i] = a[i] / m;
      for (int i = 0; i < W; ++i)
        for (int j = i; j < W; ++j) cv[(size_t)i * W + j] = cv[(size_t)j * W + i] = (q[(size_t)i * W + j] - m * mu[i] * mu[j]) / (m - 1.0);
    }
  }
  return MRGAN_OK;
}

int64_t mrgan_kernel_launches(const mrgan_handle* h) { return h ? h->launches : -1; }
double mrgan_last_device_ms(const mrgan_handle* h) { return h ? h->last_ms : -1.0; }

}  // extern "C"
