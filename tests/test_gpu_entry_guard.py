"""GPU tier of the C-ABI's error contract: every handle-taking entry point against each precondition it has -- a null
handle, a fold index of -1 and of n_folds, a handle of the wrong model, a fold before mrgan_load_fold, an SVM before
mrgan_svm_fit, a null output, an out-of-range count or label, and a data-parallel handle with virtual ranks.  Each case
checks the status and a key phrase of mrgan_last_error.  The checks run in one fixed order (handle and fold, model, the
call's own arguments, data-parallel mode and readiness), so a call that fails several of them reports the first."""
import ctypes as C

import numpy as np
import pytest

from mr_gan_b200 import _lib
from mr_gan_b200.engine import FoldGroup

pytestmark = pytest.mark.gpu

ARG, STATE = -1, -4
D, NTR, NTE, K = 16, 100, 20, 6


def _data(seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((NTR, D)).astype(np.float32), (np.arange(NTR) % K).astype(np.int32),
            rng.standard_normal((NTE, D)).astype(np.float32), (np.arange(NTE) % K).astype(np.int32))


@pytest.fixture(scope="module")
def handles():
    """G / N / S: one unloaded GAN / NN / SVM fold; Gl / Nl / Sl: the same, loaded (the SVM not fitted); V: a GAN handle
    whose two loaded folds play virtual data-parallel ranks."""
    x = _data(0)
    gs = {"G": FoldGroup([(D, NTR, NTE, 1)]), "Gl": FoldGroup([(D, NTR, NTE, 1)]),
          "N": FoldGroup([(D, NTR, NTE, 1)], model="nn"), "Nl": FoldGroup([(D, NTR, NTE, 1)], model="nn"),
          "S": FoldGroup([(D, NTR, NTE, 1)], model="svm"), "Sl": FoldGroup([(D, NTR, NTE, 1)], model="svm"),
          "V": FoldGroup([(D, NTR, NTE, 5)] * 2, batch=20)}
    for k in ("Gl", "Nl", "Sl"):
        gs[k].load_fold(0, *x)
    gs["V"].dp_init_virtual(2)
    for r in range(2):
        gs["V"].load_fold(r, *x)
    yield {k: fg._h for k, fg in gs.items()}
    for fg in gs.values():
        fg.close()


class _Bufs:
    def __init__(self):
        self._keep = []
        self.F = self._f(np.zeros(1 << 20, np.float32))          # any float input / output (a D = 16 net's Adam slot fits)
        self.ONE = self._f(np.ones(1 << 10, np.float32))         # positive C / gamma
        self.I = self._i(np.zeros(1 << 14, np.int32))            # row indices, labels, splits in range
        self.BIG = self._i(np.full(1 << 14, 1 << 20, np.int32))  # row indices / labels out of range
        self.NEG = self._i(np.full(1 << 10, -1, np.int32))       # labels / targets below 0
        self.id = C.create_string_buffer(128)

    def _f(self, a):
        self._keep.append(a)
        return _lib.fptr(a)

    def _i(self, a):
        self._keep.append(a)
        return _lib.iptr(a)


def _fold_cases(name, call, model_h, wrong_models, phrase_model):
    """null handle, fold -1 and 1 (every handle here holds one fold), and each wrong model; call(lib, h, fold, b)."""
    out = [(name + "/null", None, lambda l, h, b: call(l, h, 0, b), ARG, "null")]
    out += [(name + "/fold%d" % f, model_h, lambda l, h, b, f=f: call(l, h, f, b), ARG, "fold index out of range") for f in (-1, 1)]
    out += [(name + "/model-" + m, m, lambda l, h, b: call(l, h, 0, b), STATE, phrase_model) for m in wrong_models]
    return out


def _cases():
    c = []
    nets = "not available on an SVM handle"
    gan, nn, svm = "needs a GAN handle", "needs an NN handle", "needs an SVM handle"
    loaded, fitted, dp = "before mrgan_load_fold", "before mrgan_svm_fit", "not available on a data-parallel handle"

    def add(name, h, fn, code, phrase):
        c.append((name, h, fn, code, phrase))

    # parameters and counters
    for fn in ("set_params", "get_params"):
        call = lambda l, h, f, b, fn=fn: getattr(l, "mrgan_" + fn)(h, f, 0, b.F, l.mrgan_num_params(h, 0, 0) if h else 1)
        c += _fold_cases(fn, call, "G", ["S"], nets)
        add(fn + "/net", "N", lambda l, h, b, fn=fn: getattr(l, "mrgan_" + fn)(h, 0, 1, b.F, 1), ARG, "no such net")
        add(fn + "/length", "G", lambda l, h, b, fn=fn: getattr(l, "mrgan_" + fn)(h, 0, 0, b.F, 5), ARG, "does not match mrgan_num_params")
    c += _fold_cases("get_adam", lambda l, h, f, b: l.mrgan_get_adam(h, f, 0, b.F, b.F, 1), "G", ["S"], nets)
    add("get_adam/null-v", "G", lambda l, h, b: l.mrgan_get_adam(h, 0, 0, b.F, None, l.mrgan_num_params(h, 0, 0)), ARG, "length")
    c += _fold_cases("get_counters", lambda l, h, f, b: l.mrgan_get_counters(h, f, None, None), "G", ["S"], nets)

    # fold data
    c += _fold_cases("load_fold", lambda l, h, f, b: l.mrgan_load_fold(h, f, b.F, b.I, b.F, b.I), "G", [], "")
    add("load_fold/null", "G", lambda l, h, b: l.mrgan_load_fold(h, 0, b.F, b.I, None, b.I), ARG, "null pointer")
    add("load_fold/label", "S", lambda l, h, b: l.mrgan_load_fold(h, 0, b.F, b.I, b.F, b.BIG), ARG, "label out of range")
    add("load_dataset/null", None, lambda l, h, b: l.mrgan_load_dataset(h, 0, b.F, b.I, 4, D), ARG, "null")
    add("load_dataset/slot", "G", lambda l, h, b: l.mrgan_load_dataset(h, 8, b.F, b.I, 4, D), ARG, "bad argument")
    add("load_dataset/label", "G", lambda l, h, b: l.mrgan_load_dataset(h, 0, b.F, b.NEG, 4, D), ARG, "label out of range")
    c += _fold_cases("prepare_fold", lambda l, h, f, b: l.mrgan_prepare_fold(h, f, 0, b.I, b.I), "G", [], "")
    add("prepare_fold/slot", "N", lambda l, h, b: l.mrgan_prepare_fold(h, 0, 7, b.I, b.I), STATE, "dataset slot is empty")

    # the three step callables
    c += _fold_cases("disc_step", lambda l, h, f, b: l.mrgan_disc_step(h, f, b.F, b.I, b.F, b.F, b.F), "G", ["N", "S"], gan)
    add("disc_step/null", "G", lambda l, h, b: l.mrgan_disc_step(h, 0, b.F, b.I, b.F, b.F, None), ARG, "null pointer")
    add("disc_step/label", "G", lambda l, h, b: l.mrgan_disc_step(h, 0, b.F, b.BIG, b.F, b.F, b.F), ARG, "label out of range")
    add("disc_step/virtual", "V", lambda l, h, b: l.mrgan_disc_step(h, 0, b.F, b.I, b.F, b.F, b.F), STATE, "virtual ranks step together")
    c += _fold_cases("gen_step", lambda l, h, f, b: l.mrgan_gen_step(h, f, b.F, b.F, b.F), "G", ["N", "S"], gan)
    add("gen_step/null", "G", lambda l, h, b: l.mrgan_gen_step(h, 0, None, b.F, b.F), ARG, "null pointer")
    add("gen_step/virtual", "V", lambda l, h, b: l.mrgan_gen_step(h, 0, b.F, b.F, b.F), STATE, "virtual ranks step together")
    c += _fold_cases("test_batch", lambda l, h, f, b: l.mrgan_test_batch(h, f, b.F, b.I, 4, b.F), "G", ["S"], nets)
    add("test_batch/null", "G", lambda l, h, b: l.mrgan_test_batch(h, 0, b.F, b.I, 4, None), ARG, "null pointer")
    for n in (0, 151):        # rows of a GAN step at batch 50: 150 > n_test
        add("test_batch/n%d" % n, "G", lambda l, h, b, n=n: l.mrgan_test_batch(h, 0, b.F, b.I, n, b.F), ARG, "n exceeds")
    add("test_batch/label", "N", lambda l, h, b: l.mrgan_test_batch(h, 0, b.F, b.NEG, 4, b.F), ARG, "label out of range")

    # evaluation and epochs
    c += _fold_cases("eval", lambda l, h, f, b: l.mrgan_eval(h, f, b.F), "G", ["S"], nets)
    add("eval/null", "Gl", lambda l, h, b: l.mrgan_eval(h, 0, None), ARG, "null pointer")
    add("eval/loaded", "G", lambda l, h, b: l.mrgan_eval(h, 0, b.F), STATE, "eval " + loaded)
    add("epoch_result/null", None, lambda l, h, b: l.mrgan_epoch_result(h, None), ARG, "null")
    add("epoch_result/model-S", "S", lambda l, h, b: l.mrgan_epoch_result(h, None), STATE, nets)
    c += _fold_cases("set_epoch_rows", lambda l, h, f, b: l.mrgan_set_epoch_rows(h, f, b.I, 10, None, 0), "G", ["N", "S"], gan)
    add("set_epoch_rows/null", "G", lambda l, h, b: l.mrgan_set_epoch_rows(h, 0, None, 10, None, 0), ARG, "n_lab")
    add("set_epoch_rows/range", "G", lambda l, h, b: l.mrgan_set_epoch_rows(h, 0, b.BIG, 10, None, 0), ARG, "row out of range")
    add("train_epoch_seeded/null", None, lambda l, h, b: l.mrgan_train_epoch_seeded(h, 0, None), ARG, "null")
    for m in ("N", "S"):
        add("train_epoch_seeded/model-" + m, m, lambda l, h, b: l.mrgan_train_epoch_seeded(h, 0, None), STATE, gan)
    add("train_epoch_seeded/loaded", "G", lambda l, h, b: l.mrgan_train_epoch_seeded(h, 0, None), STATE, "train_epoch_seeded " + loaded)
    c += _fold_cases("debug_epoch_indices", lambda l, h, f, b: l.mrgan_debug_epoch_indices(h, f, b.I), "G", ["S"], nets)
    add("debug_epoch_indices/null", "G", lambda l, h, b: l.mrgan_debug_epoch_indices(h, 0, None), ARG, "null pointer")
    add("train_epoch/null", None, lambda l, h, b: l.mrgan_train_epoch(h, b.I, b.I, b.I, None), ARG, "null")
    for m in ("N", "S"):
        add("train_epoch/model-" + m, m, lambda l, h, b: l.mrgan_train_epoch(h, b.I, b.I, b.I, None), STATE, gan)
    add("train_epoch/null-idx", "G", lambda l, h, b: l.mrgan_train_epoch(h, b.I, None, b.I, None), ARG, "null index array")
    add("train_epoch/loaded", "G", lambda l, h, b: l.mrgan_train_epoch(h, b.I, b.I, b.I, None), STATE, "train_epoch " + loaded)
    add("train_epoch/range", "Gl", lambda l, h, b: l.mrgan_train_epoch(h, b.I, b.BIG, b.I, None), ARG, "row index out of range")

    # the NN twins
    c += _fold_cases("mrnn_step", lambda l, h, f, b: l.mrnn_step(h, f, b.F, b.I, 4, b.F), "N", ["G", "S"], nn)
    add("mrnn_step/null", "N", lambda l, h, b: l.mrnn_step(h, 0, b.F, None, 4, b.F), ARG, "null pointer")
    for n in (0, 21):
        add("mrnn_step/n%d" % n, "N", lambda l, h, b, n=n: l.mrnn_step(h, 0, b.F, b.I, n, b.F), ARG, "n must be in [1, batch]")
    add("mrnn_step/label", "N", lambda l, h, b: l.mrnn_step(h, 0, b.F, b.BIG, 4, b.F), ARG, "label out of range")
    add("mrnn_train_epoch/null", None, lambda l, h, b: l.mrnn_train_epoch(h, b.I, 20, None), ARG, "null")
    for m in ("G", "S"):
        add("mrnn_train_epoch/model-" + m, m, lambda l, h, b: l.mrnn_train_epoch(h, b.I, 20, None), STATE, nn)
    for n in (0, 30, 120):
        add("mrnn_train_epoch/n%d" % n, "N", lambda l, h, b, n=n: l.mrnn_train_epoch(h, b.I, n, None), ARG, "n_idx must be")
    add("mrnn_train_epoch/null-idx", "N", lambda l, h, b: l.mrnn_train_epoch(h, None, 20, None), ARG, "n_idx must be")
    add("mrnn_train_epoch/loaded", "N", lambda l, h, b: l.mrnn_train_epoch(h, b.I, 20, None), STATE, "mrnn_train_epoch " + loaded)
    add("mrnn_train_epoch/range", "Nl", lambda l, h, b: l.mrnn_train_epoch(h, b.BIG, 20, None), ARG, "row index out of range")
    c += _fold_cases("mrnn_evaluate", lambda l, h, f, b: l.mrnn_evaluate(h, f, b.F), "N", ["S"], nets)
    add("mrnn_evaluate/null", "Nl", lambda l, h, b: l.mrnn_evaluate(h, 0, None), ARG, "null pointer")
    add("mrnn_evaluate/loaded", "N", lambda l, h, b: l.mrnn_evaluate(h, 0, b.F), STATE, "evaluate " + loaded)

    # utilities
    c += _fold_cases("fill_normal", lambda l, h, f, b: l.mrgan_fill_normal(h, f, 0, 0, 2, 2, 0, b.F), "G", ["S"], nets)
    add("fill_normal/null", "G", lambda l, h, b: l.mrgan_fill_normal(h, 0, 0, 0, 2, 2, 0, None), ARG, "bad argument")
    add("fill_normal/rows", "G", lambda l, h, b: l.mrgan_fill_normal(h, 0, 0, 0, 0, 2, 0, b.F), ARG, "bad argument")
    add("adam_flat/null", None, lambda l, h, b: l.mrgan_adam_flat(h, b.F, b.F, b.F, b.F, 4, 1), ARG, "null")
    add("adam_flat/model-S", "S", lambda l, h, b: l.mrgan_adam_flat(h, b.F, b.F, b.F, b.F, 4, 1), STATE, nets)
    add("adam_flat/args", "G", lambda l, h, b: l.mrgan_adam_flat(h, b.F, None, b.F, b.F, 4, 1), ARG, "bad argument")
    add("adam_flat/t", "G", lambda l, h, b: l.mrgan_adam_flat(h, b.F, b.F, b.F, b.F, 4, 0), ARG, "bad argument")
    add("time_op/null", None, lambda l, h, b: l.mrgan_time_op(h, 0, 1, b.F), ARG, "null")
    add("time_op/out", "Gl", lambda l, h, b: l.mrgan_time_op(h, 0, 1, None), ARG, "bad argument")
    add("time_op/reps", "Gl", lambda l, h, b: l.mrgan_time_op(h, 0, 0, b.F), ARG, "bad argument")
    add("time_op/svm-op", "Gl", lambda l, h, b: l.mrgan_time_op(h, 7, 1, b.F), STATE, "does not exist for this model")
    add("time_op/net-op", "Sl", lambda l, h, b: l.mrgan_time_op(h, 0, 1, b.F), STATE, "does not exist for this model")
    add("time_op/unknown-S", "Sl", lambda l, h, b: l.mrgan_time_op(h, 99, 1, b.F), ARG, "does not exist for this model")
    add("time_op/unknown-G", "Gl", lambda l, h, b: l.mrgan_time_op(h, 99, 1, b.F), ARG, "unknown op")
    add("time_op/generator", "Nl", lambda l, h, b: l.mrgan_time_op(h, 1, 1, b.F), STATE, "no generator")
    add("time_op/loaded", "G", lambda l, h, b: l.mrgan_time_op(h, 0, 1, b.F), STATE, "time_op " + loaded)
    add("time_op/fitted", "Sl", lambda l, h, b: l.mrgan_time_op(h, 7, 1, b.F), STATE, fitted)
    add("time_op/virtual", "V", lambda l, h, b: l.mrgan_time_op(h, 10, 1, b.F), STATE, dp)
    c += _fold_cases("debug_buffer", lambda l, h, f, b: l.mrgan_debug_buffer(h, f, 0, b.F, 2, 2), "G", [], "")
    add("debug_buffer/null", "G", lambda l, h, b: l.mrgan_debug_buffer(h, 0, 0, None, 2, 2), ARG, "bad argument")
    add("debug_buffer/unknown", "G", lambda l, h, b: l.mrgan_debug_buffer(h, 0, 99, b.F, 2, 2), ARG, "unknown buffer")
    add("debug_buffer/svm", "Sl", lambda l, h, b: l.mrgan_debug_buffer(h, 0, 0, b.F, 2, 2), STATE, "fold data and kernel matrices only")
    add("debug_buffer/fitted", "Sl", lambda l, h, b: l.mrgan_debug_buffer(h, 0, 60, b.F, 2, 2), STATE, fitted)
    add("debug_gemm/null", None, lambda l, h, b: l.mrgan_debug_gemm(h, 0, 2, 2, 2, b.F, b.F, b.F, 0), ARG, "null")
    add("debug_gemm/model-S", "S", lambda l, h, b: l.mrgan_debug_gemm(h, 0, 2, 2, 2, b.F, b.F, b.F, 0), STATE, nets)
    add("debug_gemm/mode", "G", lambda l, h, b: l.mrgan_debug_gemm(h, 3, 2, 2, 2, b.F, b.F, b.F, 0), ARG, "bad argument")
    add("debug_gemm/out", "G", lambda l, h, b: l.mrgan_debug_gemm(h, 0, 2, 2, 2, b.F, b.F, None, 0), ARG, "bad argument")
    add("debug_gemm_time/null", None, lambda l, h, b: l.mrgan_debug_gemm_time(h, 0, 2, 2, 2, 1, 1, b.F), ARG, "null")
    add("debug_gemm_time/model-S", "S", lambda l, h, b: l.mrgan_debug_gemm_time(h, 0, 2, 2, 2, 1, 1, b.F), STATE, nets)
    add("debug_gemm_time/groups", "G", lambda l, h, b: l.mrgan_debug_gemm_time(h, 0, 2, 2, 2, 0, 1, b.F), ARG, "bad argument")

    # data-parallel set-up
    add("dp_init/null", None, lambda l, h, b: l.mrgan_dp_init(h, 0, 2, b.id), ARG, "null")
    add("dp_init/rank", "G", lambda l, h, b: l.mrgan_dp_init(h, 2, 2, b.id), ARG, "bad rank")
    add("dp_init/world", "G", lambda l, h, b: l.mrgan_dp_init(h, 0, 9, b.id), ARG, "at most 8 ranks")
    add("dp_init/model-N", "N", lambda l, h, b: l.mrgan_dp_init(h, 0, 2, b.id), STATE, "GAN")
    add("dp_init/twice", "V", lambda l, h, b: l.mrgan_dp_init(h, 0, 2, b.id), STATE, "dp_init called twice")
    add("dp_init_virtual/null", None, lambda l, h, b: l.mrgan_dp_init_virtual(h, 2), ARG, "null")
    add("dp_init_virtual/model-S", "S", lambda l, h, b: l.mrgan_dp_init_virtual(h, 2), STATE, "GAN")
    add("dp_init_virtual/twice", "V", lambda l, h, b: l.mrgan_dp_init_virtual(h, 2), STATE, "dp_init called twice")
    add("dp_init_virtual/world", "G", lambda l, h, b: l.mrgan_dp_init_virtual(h, 2), ARG, "exactly `world` folds")
    add("dp_ipc_export/null", None, lambda l, h, b: l.mrgan_dp_ipc_export(h, b.id), ARG, "null")
    add("dp_ipc_export/out", "G", lambda l, h, b: l.mrgan_dp_ipc_export(h, None), ARG, "null")
    add("dp_ipc_open/null", None, lambda l, h, b: l.mrgan_dp_ipc_open(h, b.id, 2), ARG, "null")
    add("dp_ipc_open/handles", "G", lambda l, h, b: l.mrgan_dp_ipc_open(h, None, 2), ARG, "null")
    add("dp_ipc_open/local", "G", lambda l, h, b: l.mrgan_dp_ipc_open(h, b.id, 2), STATE, "after mrgan_dp_init")
    add("dp_ipc_open/virtual", "V", lambda l, h, b: l.mrgan_dp_ipc_open(h, b.id, 2), STATE, "after mrgan_dp_init")

    # the SVM
    for fn, call in (("svm_fit", lambda l, h, b: l.mrgan_svm_fit(h, b.I, 12, 1.0, b.ONE, 1e-3, None)),
                     ("svm_fit_folds", lambda l, h, b: l.mrgan_svm_fit_folds(h, b.I, 12, b.ONE, b.ONE, 1e-3, None)),
                     ("svm_cv", lambda l, h, b: l.mrgan_svm_cv(h, b.I, 12, b.I, 2, b.ONE, 1, b.ONE, 1, 1e-3, b.I))):
        add(fn + "/null", None, call, ARG, "null")
        for m in ("G", "N"):
            add(fn + "/model-" + m, m, call, STATE, svm)
        add(fn + "/loaded", "S", call, STATE, "mrgan_load_fold")
    add("svm_fit/args", "Sl", lambda l, h, b: l.mrgan_svm_fit(h, None, 12, 1.0, b.ONE, 1e-3, None), ARG, "bad argument")
    add("svm_fit/C", "Sl", lambda l, h, b: l.mrgan_svm_fit(h, b.I, 12, 0.0, b.ONE, 1e-3, None), ARG, "C must be positive")
    add("svm_fit/gamma", "Sl", lambda l, h, b: l.mrgan_svm_fit_folds(h, b.I, 12, b.ONE, b.F, 1e-3, None), ARG, "gamma must be positive")
    add("svm_fit/rows", "Sl", lambda l, h, b: l.mrgan_svm_fit(h, b.BIG, 12, 1.0, b.ONE, 1e-3, None), ARG, "labeled row out of range")
    add("svm_cv/splits", "Sl", lambda l, h, b: l.mrgan_svm_cv(h, b.I, 12, b.I, 1, b.ONE, 1, b.ONE, 1, 1e-3, b.I), ARG, "n_splits >= 2")
    add("svm_cv/split", "Sl", lambda l, h, b: l.mrgan_svm_cv(h, b.I, 12, b.BIG, 2, b.ONE, 1, b.ONE, 1, 1e-3, b.I), ARG, "split index outside")
    add("svm_cv/out", "Sl", lambda l, h, b: l.mrgan_svm_cv(h, b.I, 12, b.I, 2, b.ONE, 1, b.ONE, 1, 1e-3, None), ARG, "bad argument")
    for fn in ("svm_eval", "svm_decision"):
        call = lambda l, h, f, b, fn=fn: getattr(l, "mrgan_" + fn)(h, f, b.F)
        c += _fold_cases(fn, call, "Sl", ["G", "N"], svm)
        add(fn + "/null", "Sl", lambda l, h, b, fn=fn: getattr(l, "mrgan_" + fn)(h, 0, None), ARG, "null pointer")
        add(fn + "/fitted", "Sl", lambda l, h, b, fn=fn: getattr(l, "mrgan_" + fn)(h, 0, b.F), STATE, fn + " " + fitted)

    # predictions, input gradients and saliency
    c += _fold_cases("predict", lambda l, h, f, b: l.mrgan_predict(h, f, b.I, None), "G", [], "")
    add("predict/null", "Gl", lambda l, h, b: l.mrgan_predict(h, 0, None, None), ARG, "null pointer")
    c += _fold_cases("predict_rows", lambda l, h, f, b: l.mrgan_predict_rows(h, f, b.F, 1, b.I, None), "G", [], "")
    add("predict_rows/null", "Gl", lambda l, h, b: l.mrgan_predict_rows(h, 0, None, 1, b.I, None), ARG, "null pointer")
    for n in (0, NTE + 1):
        add("predict_rows/n%d" % n, "Sl", lambda l, h, b, n=n: l.mrgan_predict_rows(h, 0, b.F, n, b.I, None), ARG, "n must be in")
    add("confusion/null", None, lambda l, h, b: l.mrgan_confusion(h, b.I), ARG, "null")
    add("confusion/out", "Gl", lambda l, h, b: l.mrgan_confusion(h, None), ARG, "null pointer")
    for fn, call in (("predict", lambda l, h, b: l.mrgan_predict(h, 0, b.I, b.F)),
                     ("predict_rows", lambda l, h, b: l.mrgan_predict_rows(h, 0, b.F, 2, b.I, b.F)),
                     ("confusion", lambda l, h, b: l.mrgan_confusion(h, b.I))):
        add(fn + "/loaded-G", "G", call, STATE, fn + " " + loaded)
        add(fn + "/loaded-N", "N", call, STATE, fn + " " + loaded)
        add(fn + "/fitted", "Sl", call, STATE, fn + " " + fitted)
        add(fn + "/virtual", "V", call, STATE, fn + ": " + dp)
    c += _fold_cases("input_grad", lambda l, h, f, b: l.mrgan_input_grad(h, f, b.F, 1, None, b.F), "G", ["S"], nets)
    add("input_grad/null", "Gl", lambda l, h, b: l.mrgan_input_grad(h, 0, b.F, 1, None, None), ARG, "null pointer")
    for n in (0, NTE + 1):
        add("input_grad/n%d" % n, "Gl", lambda l, h, b, n=n: l.mrgan_input_grad(h, 0, b.F, n, None, b.F), ARG, "n must be in")
    add("input_grad/resident", "Gl", lambda l, h, b: l.mrgan_input_grad(h, 0, None, 3, None, b.F), ARG, "resident test set")
    add("input_grad/target", "Nl", lambda l, h, b: l.mrgan_input_grad(h, 0, b.F, 2, b.NEG, b.F), ARG, "target class out of range")
    add("input_grad/loaded", "N", lambda l, h, b: l.mrgan_input_grad(h, 0, b.F, 2, None, b.F), STATE, "input_grad " + loaded)
    add("input_grad/virtual", "V", lambda l, h, b: l.mrgan_input_grad(h, 0, b.F, 2, None, b.F), STATE, "input_grad: " + dp)
    add("saliency/null", None, lambda l, h, b: l.mrgan_saliency(h, b.F), ARG, "null")
    add("saliency/model-S", "Sl", lambda l, h, b: l.mrgan_saliency(h, b.F), STATE, nets)
    add("saliency/out", "Gl", lambda l, h, b: l.mrgan_saliency(h, None), ARG, "null pointer")
    add("saliency/loaded", "G", lambda l, h, b: l.mrgan_saliency(h, b.F), STATE, "saliency " + loaded)
    add("saliency/virtual", "V", lambda l, h, b: l.mrgan_saliency(h, b.F), STATE, "saliency: " + dp)
    add("sync/null", None, lambda l, h, b: l.mrgan_sync(h), ARG, "null")
    return c


CASES = _cases()


@pytest.mark.parametrize("name,which,call,code,phrase", CASES, ids=[c[0] for c in CASES])
def test_entry_point_rejects(handles, name, which, call, code, phrase):
    lib = _lib.load()
    h = handles[which] if which else None
    got = call(lib, h, _Bufs())
    msg = lib.mrgan_last_error(h).decode()
    assert got == code, "%s: status %d (%s)" % (name, got, msg)
    assert phrase in msg, "%s: %r" % (name, msg)


def test_rejected_calls_leave_the_handles_usable(handles):
    """After every rejected call above, the loaded handles still evaluate and report no stale error."""
    lib = _lib.load()
    out = np.zeros(4, np.float32)
    assert lib.mrgan_eval(handles["Gl"], 0, _lib.fptr(out)) == 0
    assert lib.mrgan_sync(handles["V"]) == 0 and lib.mrgan_sync(handles["Sl"]) == 0
