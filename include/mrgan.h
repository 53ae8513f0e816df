/*
 * mrgan.h -- C-ABI of the B200-native replacement for mr-gan's compiled training step.
 *
 * What it replaces (reference = Healthcare-Robotics/mr-gan, paths relative to it):
 *   the three opaque callables that Keras builds with K.function at
 *   mr_gan.py:169-171 (train_batch_disc / train_batch_gen / test_batch), the
 *   inner epoch loop that drives them (mr_gan.py:183-230) and mr_nn's
 *   model.fit / model.evaluate pair (mr_nn.py:114-118).  SURVEY.md section 8(b).  mr_svm.py's
 *   SVC(kernel='rbf', C).fit / .predict (mr_svm.py:106) on the same resident fold data.
 *
 * Conventions
 *   - plain C types only; every matrix is row-major float32, labels/indices int32;
 *   - every entry point returns 0 on success, a negative mrgan_status otherwise;
 *     mrgan_last_error() gives the message (reference behaviour: a Python
 *     exception that aborts the sweep, e.g. the B==50 assumption at mr_gan.py:146);
 *   - a handle owns ALL device memory (parameters, Adam slots, activations, fold
 *     data, RNG counters) of a GROUP of folds that train side by side on one
 *     GPU; host pointers are borrowed for the duration of the call only;
 *   - a handle is bound to one CUDA device and one stream and is not thread-safe;
 *   - there is no CPU fallback: without an sm_100 device mrgan_create fails.
 *
 * Parameter vectors use the reference's weight order (Keras `trainable_weights`):
 *   discriminator (net 0): W1[D,1000] b1 W2[1000,500] b2 W3[500,250] b3
 *                          W4[250,250] b4 W5[250,250] b5 W6[250,K] b6   (mr_gan.py:117-128)
 *   generator     (net 1): W1[100,500] b1 gamma[500] beta[500] W2[500,500] b2
 *                          W3[500,D] b3                                  (mr_gan.py:110-114)
 */
#ifndef MRGAN_H_
#define MRGAN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mrgan_handle mrgan_handle;

typedef enum {
  MRGAN_OK = 0,
  MRGAN_ERR_ARG = -1,      /* bad argument / shape mismatch */
  MRGAN_ERR_CUDA = -2,     /* CUDA runtime error (message has the detail) */
  MRGAN_ERR_NO_DEVICE = -3,/* no sm_100 device: there is no CPU fallback */
  MRGAN_ERR_STATE = -4     /* call made in the wrong state (e.g. epoch before load_fold) */
} mrgan_status;

enum { MRGAN_NET_D = 0, MRGAN_NET_G = 1 };
enum { MRGAN_MODEL_GAN = 0,   /* mr_gan.py: G + D, feature matching          */
       MRGAN_MODEL_NN = 1,    /* mr_nn.py: D as a plain classifier, MSE loss */
       MRGAN_MODEL_SVM = 2 }; /* mr_svm.py: RBF C-SVC, one-vs-one (fold data + SVM workspace only: no nets) */
enum { MRGAN_PREC_FP32 = 0,   /* FFMA kernels, fp32 operands (parity mode)                  */
       MRGAN_PREC_TF32 = 1,   /* tcgen05 kind::tf32 tensor-core kernels, fp32 accumulate    */
       MRGAN_PREC_F16 = 2 };  /* tcgen05 kind::f16 on 16-bit operand COPIES: fp16 weights and activations (the same
                                 10-bit mantissa as tf32, rounded to nearest), fp16 gradients times a loss scale
                                 (4096, saturating; MRGAN_LOSS_SCALE overrides it); fp32 master weights, fp32
                                 accumulation and Adam. */

/* Hyper-parameters; mrgan_default_config() fills the reference's values. */
typedef struct {
  int model;             /* MRGAN_MODEL_*                                     */
  int n_folds;           /* folds trained side by side by this handle         */
  int batch;             /* 50 (mr_gan.py:78) / 20 (mr_nn.py:117)             */
  int n_classes;         /* 6  (mr_gan.py:80)                                 */
  int noise_dim;         /* 100 (mr_gan.py:77)                                */
  int precision;         /* MRGAN_PREC_*                                      */
  int shared_t;          /* 1: D and G share Adam's step counter (mr_gan.py:165-167) */
  int eval_each_epoch;   /* 1: batch-wise test error every epoch (mr_gan.py:219-223) */
  int device;            /* CUDA device ordinal                               */
  float lr, beta1, beta2, adam_eps;   /* 6e-4, .5, .999, 1e-8 (mr_gan.py:165) */
  float bn_eps;          /* 2e-5 (mr_gan.py:112)                              */
  float unlabeled_weight;/* 1 (mr_gan.py:79)                                  */
  float sigma_in, sigma_hidden; /* .3, .5 (mr_gan.py:118-126)                 */
  /* discriminator variants of others/wganlpctsemi.py:166-179 (defaults reproduce mr_gan.py / mr_nn.py): */
  int hidden_act;        /* MRGAN_ACT_RELU (mr_gan.py:119-127) or MRGAN_ACT_LEAKY_RELU                 */
  float leaky_alpha;     /* LeakyReLU slope, 0.3 = Keras default (wganlpctsemi.py:169)                 */
  float dropout;         /* > 0: Dropout(rate) in front of hidden layers 2..5 in place of their
                            GaussianNoise (wganlpctsemi.py:170); 0: GaussianNoise(sigma_hidden)        */
} mrgan_config;
enum { MRGAN_ACT_RELU = 0, MRGAN_ACT_LEAKY_RELU = 1 };

typedef struct {
  int D;                 /* input width of this fold (X_train.shape[1])       */
  int n_train;           /* rows of X_train (must be equal for all folds of a handle) */
  int n_test;            /* rows of X_test                                    */
  uint64_t seed;         /* Philox key of this fold's noise streams           */
} mrgan_fold_shape;

/* statistics of one epoch and one fold (mr_gan.py:215-223) */
typedef struct {
  float loss_lab, loss_unl, train_err, loss_gen;  /* means over the epoch's batches */
  float test_err;        /* mean batch-wise test error (-1 if eval_each_epoch == 0)  */
} mrgan_epoch_stats;

int  mrgan_default_config(int model, mrgan_config* cfg);

/* Replaces model construction + K.function compilation, mr_gan.py:109-171. */
int  mrgan_create(const mrgan_config* cfg, const mrgan_fold_shape* folds, mrgan_handle** out);
int  mrgan_destroy(mrgan_handle* h);
const char* mrgan_last_error(const mrgan_handle* h);   /* h may be NULL (creation errors) */
int  mrgan_sync(mrgan_handle* h);

/* Theano shared variables of the nets (mr_gan.py:131-133): read / write, reference order. */
int64_t mrgan_num_params(const mrgan_handle* h, int fold, int net);
int  mrgan_set_params(mrgan_handle* h, int fold, int net, const float* src, int64_t n);
int  mrgan_get_params(mrgan_handle* h, int fold, int net, float* dst, int64_t n);
/* Adam slots m, v (Keras optimizer weights) and the step counters, for tests / checkpoints. */
int  mrgan_get_adam(mrgan_handle* h, int fold, int net, float* m, float* v, int64_t n);
int  mrgan_get_counters(mrgan_handle* h, int fold, int* iterations, int* rng_step);

/* Fold data made device-resident once (replaces the per-call numpy slices of
 * mr_gan.py:207,213,222): scaled X_train/X_test, labels. */
int  mrgan_load_fold(mrgan_handle* h, int fold,
                     const float* x_train, const int32_t* y_train,
                     const float* x_test, const int32_t* y_test);

/* Device-side fold preparation (SURVEY.md 8(f)-2; replaces the host work of mr_gan.py:96-101 and the per-fold upload):
 * the raw feature matrix of a sweep is uploaded ONCE per handle (all folds of a table share it, mr_gan.py:250-257);
 * a fold is then cut on the device from row indices: StandardScaler statistics over its training rows (float64
 * accumulation, population variance, zero-variance guard, like sklearn), scaled X_train in the given (already shuffled)
 * order, scaled X_test, gathered labels.  slot < 8. */
int  mrgan_load_dataset(mrgan_handle* h, int slot, const float* x, const int32_t* y, int n_rows, int D);
int  mrgan_prepare_fold(mrgan_handle* h, int fold, int slot, const int32_t* train_rows, const int32_t* test_rows);

/* The three K.function callables, one fold at a time, HOST buffers:
 *   train_batch_disc([1, x_lab, labels, x_unl, noise]) -> [loss_lab, loss_unl, train_err]  mr_gan.py:169
 *   train_batch_gen ([1, x_unl, noise])               -> loss_gen                          mr_gan.py:170
 *   test_batch      ([0, x, labels])                  -> err                               mr_gan.py:171
 * rows = cfg.batch for the two train calls; n <= max(n_test, 3*batch) for test_batch. */
int  mrgan_disc_step(mrgan_handle* h, int fold, const float* x_lab, const int32_t* labels,
                     const float* x_unl, const float* z, float out[3]);
int  mrgan_gen_step(mrgan_handle* h, int fold, const float* x_unl, const float* z, float out[1]);
int  mrgan_test_batch(mrgan_handle* h, int fold, const float* x, const int32_t* y, int n, float* err);

/* The epoch loop of mr_gan.py:183-223 for ALL folds of the handle as one CUDA
 * graph launch: n_train/batch x (D step, G step), then the batch-wise test pass.
 * idx_* are this epoch's row indices into X_train ([n_folds][n_train], the
 * permutations of mr_gan.py:189-202).  stats may be NULL (asynchronous; collect
 * with mrgan_epoch_result). */
int  mrgan_train_epoch(mrgan_handle* h, const int32_t* idx_lab, const int32_t* idx_unl,
                       const int32_t* idx_unl2, mrgan_epoch_stats* stats);
int  mrgan_epoch_result(mrgan_handle* h, mrgan_epoch_stats* stats);
/* The same epoch with the permutations of mr_gan.py:189-202 drawn ON THE DEVICE (SURVEY.md 8(f)-2): the host sends an
 * epoch number instead of 3 x int32[n_train] per fold.  mrgan_set_epoch_rows uploads, once per fold, the labeled rows
 * (mr_gan.py:102) and the optional unlabeled subset of table 6 (mr_gan.py:107; NULL / 0 = all training rows); every
 * epoch then tiles fresh permutations of them exactly like the reference (floor(N/L) permutations of the L rows plus a
 * permutation of the first N mod L), keyed by (fold seed, epoch, stream).  Subsets of at most 8192 rows. */
int  mrgan_set_epoch_rows(mrgan_handle* h, int fold, const int32_t* lab_rows, int n_lab, const int32_t* unl_rows, int n_unl);
int  mrgan_train_epoch_seeded(mrgan_handle* h, uint32_t epoch, mrgan_epoch_stats* stats);
/* test hook: the three index streams of the last epoch, [3][n_train] */
int  mrgan_debug_epoch_indices(mrgan_handle* h, int fold, int32_t* dst);
/* testerror on the full resident test set in one call, mr_gan.py:230 */
int  mrgan_eval(mrgan_handle* h, int fold, float* err);

/* Data-parallel large-batch mode (BASELINE.json config 5; the reference's batch is fixed at 50, mr_gan.py:78, so this
 * is an extension): W processes, one GPU each, hold replicas of ONE set of folds; cfg.batch is the LOCAL batch, the
 * global batch is W * cfg.batch.  After mrgan_dp_init every train call all-reduces (NCCL, in-stream, over
 * NVLink / NVSwitch) the BatchNorm and feature-matching batch statistics and the flat gradient, so the W ranks
 * compute exactly the single-GPU step at the global batch, including its noise stream.  Each rank passes its own
 * slice of the global batch (rows [rank*batch, (rank+1)*batch) of every section).
 *   mrgan_nccl_unique_id: 128 bytes from ncclGetUniqueId (call on rank 0, broadcast with any host transport). */
int  mrgan_nccl_unique_id(void* id128);
int  mrgan_dp_init(mrgan_handle* h, int rank, int world, const void* id128);
/* Fused gradient exchange over NVLink peer memory (csrc/kernels_dp.cuh): after mrgan_dp_init every rank exports 128 bytes
 * (CUDA IPC handles of its arenas), the host exchanges them with any transport, and every rank opens all of them.  From
 * then on the per-step exchange is ONE kernel per rank -- reduce-scatter of the flat gradient by peer loads, Adam on the
 * owned 1/W shard, all-gather of the updated weights by peer stores -- instead of ncclAllReduce + a full-size Adam
 * (which remains the path when the handles are not opened).
 *   handles: world x 128 bytes, rank-major. */
int  mrgan_dp_ipc_export(mrgan_handle* h, void* out128);
int  mrgan_dp_ipc_open(mrgan_handle* h, const void* handles, int world);
/* The same data-parallel path with VIRTUAL ranks on one GPU (test / single-GPU validation of everything but the
 * transport): the handle must hold exactly `world` folds of identical shape and noise key; fold r plays rank r
 * (its resident rows are rank r's slice of the global batch) and every collective is a rank-ordered local sum over
 * the folds' buffers.  Train with mrgan_train_epoch; the per-fold step calls are rejected in this mode. */
int  mrgan_dp_init_virtual(mrgan_handle* h, int world);

/* mr_nn.py:114-118 twins (handle created with MRGAN_MODEL_NN):
 *   one model.fit batch: x[n,D], labels[n] -> {mse loss, accuracy}; n <= batch */
int  mrnn_step(mrgan_handle* h, int fold, const float* x, const int32_t* labels, int n, float out[2]);
/* one fit epoch over idx ([n_folds][n_idx] rows of X_train, n_idx % batch == 0), all folds */
int  mrnn_train_epoch(mrgan_handle* h, const int32_t* idx, int n_idx, float* loss_acc /* [n_folds][2] or NULL */);
/* model.evaluate(X_test, y_test) -> {mse loss, accuracy} */
int  mrnn_evaluate(mrgan_handle* h, int fold, float out[2]);

/* mr_svm.py:106 SVC(kernel='rbf', C).fit(x_labeled, y_labeled) for ALL folds of the handle (created with MRGAN_MODEL_SVM),
 * libsvm's solver (sklearn/svm/src/libsvm/svm.cpp) without shrinking; then the prediction of every fold's full resident X_test.
 *   lab_rows [n_folds][n_lab]: rows of the resident X_train, class-major (labels non-decreasing); gamma [n_folds];
 *   tol: libsvm eps.  A class pair has at most 8192 rows.
 *   n_iter [n_folds][K(K-1)/2] or NULL; returns MRGAN_ERR_STATE if a pair hit the iteration cap max(1e7, 100 n). */
int  mrgan_svm_fit(mrgan_handle* h, const int32_t* lab_rows, int n_lab, float C, const float* gamma, float tol, int32_t* n_iter);
/* mrgan_svm_fit with its own C per fold: C [n_folds] (mrgan_svm_fit is this call with C broadcast). */
int  mrgan_svm_fit_folds(mrgan_handle* h, const int32_t* lab_rows, int n_lab, const float* C, const float* gamma, float tol,
                         int32_t* n_iter);
/* The inner cross-validation of GridSearchCV(SVC(kernel='rbf', tol), {'C': C, 'gamma': gamma}, cv) for every fold: one SVC fit
 * per (fold, gamma, C, split) on the split's inner-training rows (labeled rows with split index != s, in the labeled order),
 * voted on its validation rows (split index == s).  Same labeled rows and checks as mrgan_svm_fit; also
 *   split [n_folds][n_lab] in [0, n_splits), n_splits >= 2, every split with a validation row and every class among its
 *   inner-training rows; C [nC] > 0; gamma [n_folds][nG] > 0 (absolute); otherwise MRGAN_ERR_ARG.
 *   wrong [n_folds][nG][nC][n_splits]: misclassified validation rows (integers, bitwise reproducible).
 * One gamma column at a time in the fit's labeled x labeled buffers.  MRGAN_ERR_STATE if a problem hits the iteration cap (the
 * message names fold, gamma, C, split and class pair).  A call that passes the argument checks invalidates a previous fit:
 * mrgan_svm_eval, mrgan_svm_decision, mrgan_predict*, mrgan_confusion and the SVM phases of mrgan_time_op return
 * MRGAN_ERR_STATE until the next mrgan_svm_fit*.  A call rejected with MRGAN_ERR_ARG leaves the previous fit valid. */
int  mrgan_svm_cv(mrgan_handle* h, const int32_t* lab_rows, int n_lab, const int32_t* split, int n_splits, const float* C, int nC,
                  const float* gamma, int nG, float tol, int32_t* wrong);
int  mrgan_svm_eval(mrgan_handle* h, int fold, float* err);                 /* full resident X_test, ovo vote */
int  mrgan_svm_decision(mrgan_handle* h, int fold, float* dst);             /* test hook: [n_test][K(K-1)/2] */

/* Predictions of a trained fold (GAN / NN: the current weights, the phase-0 forward of mrgan_eval; SVM: after mrgan_svm_fit).
 * The predicted class is the first maximal logit (GAN / NN; the rule behind the error of mrgan_eval) or libsvm's one-vs-one
 * vote, the first class with the most votes (SVM).  Scores are raw: logits, or decision values, not probabilities.
 *   mrgan_predict: the fold's resident test set: pred [n_test]; scores [n_test][K] logits (GAN / NN)
 *     or [n_test][K(K-1)/2] decision values (SVM, pairs (0,1),(0,2),...); scores may be NULL.
 *   mrgan_predict_rows: rows x [n][D_fold] in the fold's SCALED input space (that of mrgan_test_batch and of the resident
 *     X_test), 1 <= n <= n_test of the fold; same outputs.  Leaves every later result on the resident test set unchanged.
 *   mrgan_confusion: every fold of the handle in one pass over its resident test set: out [n_folds][K][K] int32 counts,
 *     rows = true class, columns = predicted class.
 * MRGAN_ERR_ARG: null pred / x / out, fold or n out of range.  MRGAN_ERR_STATE: a GAN / NN fold not loaded, an SVM handle
 * before mrgan_svm_fit, or a data-parallel handle (mrgan_dp_init / mrgan_dp_init_virtual).  Like mrgan_eval, each call first
 * completes a pending asynchronous epoch, whose statistics it leaves unchanged. */
int  mrgan_predict(mrgan_handle* h, int fold, int32_t* pred, float* scores);
int  mrgan_predict_rows(mrgan_handle* h, int fold, const float* x, int n, int32_t* pred, float* scores);
int  mrgan_confusion(mrgan_handle* h, int32_t* out);

/* Input gradients of a trained GAN / NN fold (the activation maps of the reference's others/mr_nn_activation_map.py):
 *   grad[r][j] = d log softmax(l(x_r))[t_r] / d x_r[j], l = the phase-0 logits of mrgan_predict, x in the fold's SCALED space.
 *   x: rows [n][D_fold], or NULL = the fold's resident X_test (then n must equal its n_test); 1 <= n <= n_test
 *   target: [n] classes in [0, K), or NULL = each row's predicted class (first maximal logit)
 *   grad: [n][D_fold] */
int  mrgan_input_grad(mrgan_handle* h, int fold, const float* x, int n, const int32_t* target, float* grad);
/* Every fold of the handle in one pass over its resident test set, target = the true class:
 *   profile [n_folds][K][D_max] = mean over the test rows of true class c of |grad[r][j]|; 0 beyond a fold's D and for a
 *   class without test rows.  Fixed summation order: bitwise reproducible and independent of the grouping.
 * MRGAN_ERR_ARG: null grad / profile, fold or n out of range, x == NULL with n != n_test, a target outside [0, K).
 * MRGAN_ERR_STATE: an SVM handle, a fold not loaded, or a data-parallel handle.  Like mrgan_predict, each call first completes
 * a pending asynchronous epoch, whose statistics it leaves unchanged, and changes no later result of the handle. */
int  mrgan_saliency(mrgan_handle* h, float* profile);

/* Utilities used by tests and bench */
int  mrgan_fill_normal(mrgan_handle* h, int fold, int step, int tensor_id, int rows, int cols,
                       int row0, float* dst /* host [rows, cols] */);
int  mrgan_adam_flat(mrgan_handle* h, float* p, float* m, float* v, const float* g, int64_t n,
                     int t /* 1-based */);              /* host buffers; fused flat Adam, SURVEY a8 */
/* Average device time (CUDA events on the handle's stream) of `reps` back-to-back launches of one
 * kernel of the step over ALL folds of the handle -- the live roofline probe bench.py uses.
 * Mutates the training state (run it after the measured region). */
enum { MRGAN_TIME_ADAM_D = 0, MRGAN_TIME_ADAM_G = 1, MRGAN_TIME_DW1 = 2, MRGAN_TIME_FWD1 = 3,
       MRGAN_TIME_DISC_STEP = 4, MRGAN_TIME_GEN_STEP = 5,
       MRGAN_TIME_DX1 = 6,     /* dFake = dZ1 W1^T of the generator step: the dX pass over the widest layer */
       /* SVM handles, after mrgan_svm_fit (re-running a phase reproduces its results bitwise): */
       MRGAN_TIME_SVM_KMAT = 7,     /* both kernel matrices of all folds (operand split + tcgen05 GEMM + RBF) */
       MRGAN_TIME_SVM_SMO = 8,      /* the SMO solver of every (fold, class pair) */
       MRGAN_TIME_SVM_PREDICT = 9, /* decision values, vote and error count of every test row */
       /* GAN / NN handles, read-only (the training state is unchanged): */
       MRGAN_TIME_SALIENCY = 10 }; /* mrgan_saliency's pass: eval forward, seed, dX chain and profile of every fold */
int  mrgan_time_op(mrgan_handle* h, int which, int reps, float* ms_avg);
/* Debug/test hook: copy an intermediate buffer of the last step of one fold to the host
 * (dst is [rows, cols] dense).  which: 0..5 = noisy layer inputs a[l], 10+l = post-ReLU h[l],
 * 20+l = dZ[l], 30 = logits, 31 = dlogits, 32 = dFake, 40 = z, 41 = G h1, 42 = G BN out,
 * 43 = G h2, 44 = G dZ2, 45 = G dU, 46 = G dZ1, 50 = resident X_train, 51 = resident X_test;
 * SVM handles after mrgan_svm_fit: 60 = labeled x labeled kernel matrix [n_lab][n_lab], 61 = test x labeled [n_test][n_lab]. */
int  mrgan_debug_buffer(mrgan_handle* h, int fold, int which, float* dst, int rows, int cols);
/* Test hook: one stand-alone GEMM through the step's kernels (use_tc = 1: tcgen05 path, 0: fp32 path).
 * mode 0: C[M,N] = A[M,K] B[K,N]   mode 1: C[M,N] = A[M,K] B[N,K]^T   mode 2: C[M,N] = A[K,M]^T B[K,N]
 * Dense row-major host arrays. */
int  mrgan_debug_gemm(mrgan_handle* h, int mode, int M, int N, int K, const float* A, const float* B, float* C, int use_tc);
/* Test hook: average device ms of `reps` launches of the stand-alone GEMM above on zero-filled operands,
 * replicated over `groups` independent problems (grid.z), tcgen05 path. */
int  mrgan_debug_gemm_time(mrgan_handle* h, int mode, int M, int N, int K, int groups, int reps, float* ms);
int64_t mrgan_kernel_launches(const mrgan_handle* h); /* kernels launched so far (graph nodes count per replay) */
double  mrgan_last_device_ms(const mrgan_handle* h);  /* CUDA-event time of the last train_epoch */
const char* mrgan_version(void);
/* ABI guard for hand-written bindings (ctypes / cgo / JNI lay the structs out by hand): fills
 * {MRGAN_ABI_VERSION, sizeof(mrgan_config), sizeof(mrgan_fold_shape), sizeof(mrgan_epoch_stats)}. */
#define MRGAN_ABI_VERSION 3
int  mrgan_abi_info(int out[4]);

#ifdef __cplusplus
}
#endif
#endif /* MRGAN_H_ */
