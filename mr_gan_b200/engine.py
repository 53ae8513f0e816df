"""Host-side mirror of the reference's compiled training functions.

``FoldGroup`` owns one ``mrgan_handle`` (include/mrgan.h): a group of folds that train
side by side on one B200.  Its methods mirror, per fold, the three callables Keras
builds at mr_gan.py:169-171 (same argument order and return values) plus the
epoch-at-once call that replaces the Python loop of mr_gan.py:204-223.

PyTorch is not needed here; numpy arrays cross the C-ABI as plain pointers.
"""
import ctypes as C

import numpy as np

from . import _lib
from .model import disc_shapes, gen_shapes

MODEL = {"gan": 0, "nn": 1, "svm": 2}
PRECISION = {"fp32": 0, "tf32": 1, "f16": 2}      # f16 (the trainers' and CLIs' default): fp16 operand copies, fp32 master weights / accumulation


class MrganError(RuntimeError):
    pass


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class FoldGroup:
    def __init__(self, shapes, model="gan", precision="fp32", device=0, batch=None, n_classes=6,
                 eval_each_epoch=True, shared_t=True, **hyper):
        """shapes: iterable of (D, n_train, n_test, seed) -- one entry per fold of the group."""
        self.lib = _lib.load()
        cfg = _lib.Config()
        self._chk(self.lib.mrgan_default_config(MODEL[model], C.byref(cfg)), None)
        shapes = list(shapes)
        cfg.n_folds = len(shapes)
        cfg.precision = PRECISION[precision]
        cfg.device = int(device)
        cfg.n_classes = int(n_classes)
        cfg.eval_each_epoch = int(bool(eval_each_epoch))
        cfg.shared_t = int(bool(shared_t))
        if batch is not None:
            cfg.batch = int(batch)
        for k, v in hyper.items():
            if not hasattr(cfg, k):
                raise TypeError("unknown hyper-parameter %r" % k)
            setattr(cfg, k, v)
        self.cfg = cfg
        self.model = model
        self.n_folds = len(shapes)
        self.shapes = [(int(D), int(ntr), int(nte), int(seed)) for D, ntr, nte, seed in shapes]
        arr = (_lib.FoldShape * self.n_folds)()
        for i, (D, ntr, nte, seed) in enumerate(self.shapes):
            arr[i].D, arr[i].n_train, arr[i].n_test, arr[i].seed = D, ntr, nte, seed & 0xFFFFFFFFFFFFFFFF
        h = C.c_void_p()
        self._h = None
        self._chk(self.lib.mrgan_create(C.byref(cfg), arr, C.byref(h)), None)
        self._h = h
        self.batch = cfg.batch
        self.noise_dim = cfg.noise_dim
        self.n_train = self.shapes[0][1]

    # ------------------------------------------------------------------ data-parallel large-batch mode
    @staticmethod
    def nccl_unique_id():
        """128-byte NCCL id (rank 0 creates it, every rank passes it to dp_init)."""
        buf = C.create_string_buffer(128)
        lib = _lib.load()
        if lib.mrgan_nccl_unique_id(buf) != 0:
            raise MrganError("mrgan_nccl_unique_id: %s" % lib.mrgan_last_error(None).decode())
        return buf.raw

    def dp_init(self, rank, world, unique_id, allgather=None):
        """Join a data-parallel group: this handle's `batch` becomes the LOCAL batch (global = world * batch).

        allgather: optional callable bytes -> list of `world` bytes objects (rank order), e.g. built on
        ``torch.distributed.all_gather_object``.  When given, the ranks exchange the CUDA IPC handles of their arenas and the
        per-step gradient exchange becomes the fused peer-memory kernel (reduce-scatter + sharded Adam + all-gather);
        otherwise it is ncclAllReduce + a full Adam on every rank."""
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._chk(self.lib.mrgan_dp_init(self._h, int(rank), int(world), buf))
        self.dp_rank, self.dp_world = int(rank), int(world)
        if allgather is not None and world > 1:
            mine = C.create_string_buffer(128)
            self._chk(self.lib.mrgan_dp_ipc_export(self._h, mine))
            every = allgather(mine.raw)
            if len(every) != world or any(len(b) != 128 for b in every):
                raise ValueError("dp_init: allgather must return one 128-byte handle block per rank")
            blob = C.create_string_buffer(b"".join(every), 128 * world)
            self._chk(self.lib.mrgan_dp_ipc_open(self._h, blob, int(world)))

    def dp_init_virtual(self, world):
        """The data-parallel path with the handle's `world` folds playing the ranks on ONE GPU (collectives become
        rank-ordered local sums); fold r's resident rows are rank r's slice of the global batch."""
        self._chk(self.lib.mrgan_dp_init_virtual(self._h, int(world)))
        self.dp_rank, self.dp_world = -1, int(world)

    # ------------------------------------------------------------------ plumbing
    def _chk(self, rc, h="self"):
        if rc != 0:
            handle = self._h if h == "self" else None
            msg = self.lib.mrgan_last_error(handle)
            raise MrganError("libmrgan error %d: %s" % (rc, msg.decode() if msg else "?"))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.mrgan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def sync(self):
        self._chk(self.lib.mrgan_sync(self._h))

    # ------------------------------------------------------------------ parameters
    def _shapes(self, fold, net):
        D = self.shapes[fold][0]
        return disc_shapes(D, self.cfg.n_classes) if net == 0 else gen_shapes(D, self.noise_dim)

    def num_params(self, fold, net):
        return int(self.lib.mrgan_num_params(self._h, fold, net))

    def set_params(self, fold, net, params):
        """params: list of arrays in the reference's weight order (Keras trainable_weights)."""
        shp = self._shapes(fold, net)
        if len(params) != len(shp):
            raise ValueError("expected %d arrays" % len(shp))
        for p, s in zip(params, shp):
            if tuple(np.shape(p)) != tuple(s):
                raise ValueError("parameter shape %s != %s" % (np.shape(p), s))
        flat = _f32(np.concatenate([np.asarray(p, dtype=np.float32).ravel() for p in params]))
        self._chk(self.lib.mrgan_set_params(self._h, fold, net, _lib.fptr(flat), flat.size))

    def _split(self, flat, fold, net):
        out, o = [], 0
        for s in self._shapes(fold, net):
            n = int(np.prod(s))
            out.append(flat[o:o + n].reshape(s).copy())
            o += n
        return out

    def get_params(self, fold, net):
        flat = np.empty(self.num_params(fold, net), dtype=np.float32)
        self._chk(self.lib.mrgan_get_params(self._h, fold, net, _lib.fptr(flat), flat.size))
        return self._split(flat, fold, net)

    def get_adam(self, fold, net):
        n = self.num_params(fold, net)
        m, v = np.empty(n, dtype=np.float32), np.empty(n, dtype=np.float32)
        self._chk(self.lib.mrgan_get_adam(self._h, fold, net, _lib.fptr(m), _lib.fptr(v), n))
        return self._split(m, fold, net), self._split(v, fold, net)

    def counters(self, fold):
        it, rs = C.c_int(), C.c_int()
        self._chk(self.lib.mrgan_get_counters(self._h, fold, C.byref(it), C.byref(rs)))
        return it.value, rs.value

    # ------------------------------------------------------------------ data
    def load_fold(self, fold, x_train, y_train, x_test, y_test):
        D, ntr, nte, _ = self.shapes[fold]
        x_train, x_test = _f32(x_train), _f32(x_test)
        y_train, y_test = _i32(y_train), _i32(y_test)
        if x_train.shape != (ntr, D) or x_test.shape != (nte, D) or y_train.shape != (ntr,) or y_test.shape != (nte,):
            raise ValueError("fold %d: data does not match the declared shape (D=%d, n_train=%d, n_test=%d)"
                             % (fold, D, ntr, nte))
        self._chk(self.lib.mrgan_load_fold(self._h, fold, _lib.fptr(x_train), _lib.iptr(y_train),
                                           _lib.fptr(x_test), _lib.iptr(y_test)))

    def load_dataset(self, slot, x, y):
        """Upload the raw feature matrix of a sweep once; folds are then cut on the device (prepare_fold)."""
        x, y = _f32(x), _i32(y)
        if x.ndim != 2 or y.shape != (x.shape[0],):
            raise ValueError("load_dataset: x must be [n, D] and y [n]")
        self._chk(self.lib.mrgan_load_dataset(self._h, int(slot), _lib.fptr(x), _lib.iptr(y), x.shape[0], x.shape[1]))

    def prepare_fold(self, fold, slot, train_rows, test_rows):
        """Device-side mr_gan.py:96-101: scaler statistics over train_rows, scaled + gathered X_train (in the given,
        already shuffled order) / X_test, gathered labels."""
        D, ntr, nte, _ = self.shapes[fold]
        tr, te = _i32(train_rows), _i32(test_rows)
        if tr.shape != (ntr,) or te.shape != (nte,):
            raise ValueError("prepare_fold: expected %d train and %d test rows" % (ntr, nte))
        self._chk(self.lib.mrgan_prepare_fold(self._h, int(fold), int(slot), _lib.iptr(tr), _lib.iptr(te)))

    # ------------------------------------------------------------------ the K.function callables
    def train_batch_disc(self, fold, x_lab, labels, x_unl, noise):
        """mr_gan.py:169 ``train_batch_disc([1, x_lab, labels, x_unl, noise])``."""
        B, D = self.batch, self.shapes[fold][0]
        x_lab, x_unl, noise, labels = _f32(x_lab), _f32(x_unl), _f32(noise), _i32(labels)
        if x_lab.shape != (B, D) or x_unl.shape != (B, D) or noise.shape != (B, self.noise_dim) or labels.shape != (B,):
            raise ValueError("train_batch_disc: expected x_lab/x_unl [%d,%d], labels [%d], noise [%d,%d]"
                             % (B, D, B, B, self.noise_dim))
        out = np.zeros(3, dtype=np.float32)
        self._chk(self.lib.mrgan_disc_step(self._h, fold, _lib.fptr(x_lab), _lib.iptr(labels), _lib.fptr(x_unl),
                                           _lib.fptr(noise), _lib.fptr(out)))
        return [out[0], out[1], out[2]]

    def train_batch_gen(self, fold, x_unl, noise):
        """mr_gan.py:170 ``train_batch_gen([1, x_unl, noise])``."""
        B, D = self.batch, self.shapes[fold][0]
        x_unl, noise = _f32(x_unl), _f32(noise)
        if x_unl.shape != (B, D) or noise.shape != (B, self.noise_dim):
            raise ValueError("train_batch_gen: expected x_unl [%d,%d], noise [%d,%d]" % (B, D, B, self.noise_dim))
        out = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.mrgan_gen_step(self._h, fold, _lib.fptr(x_unl), _lib.fptr(noise), _lib.fptr(out)))
        return out[0]

    def test_batch(self, fold, x, y):
        """mr_gan.py:171 ``test_batch([0, x, labels])``."""
        x, y = _f32(x), _i32(y)
        if x.ndim != 2 or x.shape[1] != self.shapes[fold][0] or y.shape != (x.shape[0],):
            raise ValueError("test_batch: bad shapes")
        out = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.mrgan_test_batch(self._h, fold, _lib.fptr(x), _lib.iptr(y), x.shape[0], _lib.fptr(out)))
        return out[0]

    # ------------------------------------------------------------------ epoch at once
    def train_epoch(self, idx_lab, idx_unl, idx_unl2, wait=True):
        """One epoch of mr_gan.py:204-223 for every fold.  idx_*: int32 [n_folds, n_train] rows of X_train.

        Returns float32 [n_folds, 5] = loss_lab, loss_unl, train_err, loss_gen, test_err (epoch means),
        or None when wait=False (collect with epoch_result())."""
        shp = (self.n_folds, self.n_train)
        a, b, c = _i32(idx_lab), _i32(idx_unl), _i32(idx_unl2)
        if a.shape != shp or b.shape != shp or c.shape != shp:
            raise ValueError("train_epoch: index arrays must be [%d, %d]" % shp)
        self._chk(self.lib.mrgan_train_epoch(self._h, _lib.iptr(a), _lib.iptr(b), _lib.iptr(c), None))
        return self.epoch_result() if wait else None

    def set_epoch_rows(self, fold, lab_rows, unl_rows=None):
        """Device-side epoch permutations: the labeled rows (mr_gan.py:102) and the optional unlabeled subset (mr_gan.py:107)."""
        lab = _i32(lab_rows)
        unl = _i32(unl_rows) if unl_rows is not None else None
        self._chk(self.lib.mrgan_set_epoch_rows(self._h, int(fold), _lib.iptr(lab), lab.size,
                                                _lib.iptr(unl) if unl is not None else None, unl.size if unl is not None else 0))

    def train_epoch_seeded(self, epoch, wait=True):
        """One epoch with the permutations of mr_gan.py:189-202 drawn on the device from (fold seed, epoch)."""
        self._chk(self.lib.mrgan_train_epoch_seeded(self._h, int(epoch) & 0xFFFFFFFF, None))
        return self.epoch_result() if wait else None

    def epoch_indices(self, fold):
        """Test hook: the three index streams the last epoch used, int32 [3, n_train]."""
        out = np.empty((3, self.n_train), dtype=np.int32)
        self._chk(self.lib.mrgan_debug_epoch_indices(self._h, int(fold), _lib.iptr(out)))
        return out

    def epoch_result(self):
        st = (_lib.EpochStats * self.n_folds)()
        self._chk(self.lib.mrgan_epoch_result(self._h, st))
        return np.array([[s.loss_lab, s.loss_unl, s.train_err, s.loss_gen, s.test_err] for s in st], dtype=np.float32)

    def eval(self, fold):
        """mr_gan.py:230: error on the whole resident test set in one call."""
        out = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.mrgan_eval(self._h, fold, _lib.fptr(out)))
        return out[0]

    # ------------------------------------------------------------------ mr_nn twins
    def nn_step(self, fold, x, labels):
        x, labels = _f32(x), _i32(labels)
        out = np.zeros(2, dtype=np.float32)
        self._chk(self.lib.mrnn_step(self._h, fold, _lib.fptr(x), _lib.iptr(labels), x.shape[0], _lib.fptr(out)))
        return out[0], out[1]

    def nn_train_epoch(self, idx, wait=True):
        idx = _i32(idx)
        if idx.ndim != 2 or idx.shape[0] != self.n_folds:
            raise ValueError("nn_train_epoch: idx must be [n_folds, n_idx]")
        out = np.zeros((self.n_folds, 2), dtype=np.float32)
        self._chk(self.lib.mrnn_train_epoch(self._h, _lib.iptr(idx), idx.shape[1], _lib.fptr(out) if wait else None))
        return out if wait else None

    def nn_evaluate(self, fold):
        out = np.zeros(2, dtype=np.float32)
        self._chk(self.lib.mrnn_evaluate(self._h, fold, _lib.fptr(out)))
        return out[0], out[1]

    # ------------------------------------------------------------------ mr_svm (model='svm')
    @property
    def n_pairs(self):
        K = self.cfg.n_classes
        return K * (K - 1) // 2

    def _svm_lab(self, fn, lab_rows):
        lab = _i32(lab_rows)
        if lab.ndim != 2 or lab.shape[0] != self.n_folds:
            raise ValueError(fn + ": lab_rows must be [n_folds, n_lab]")
        return lab

    def svm_fit(self, lab_rows, C=1.0, gamma=None, tol=1e-3):
        """mr_svm.py:106 ``SVC(kernel='rbf', C).fit`` for every fold, then the prediction of every fold's test set.
        lab_rows: int32 [n_folds, n_lab] class-major rows of X_train; C, gamma: per-fold list / scalar (gamma None: 1 / D).
        Returns the SMO iterations, int32 [n_folds, n_pairs]."""
        lab = self._svm_lab("svm_fit", lab_rows)
        if gamma is None:
            gamma = [1.0 / D for D, _, _, _ in self.shapes]
        g = _f32(np.broadcast_to(np.asarray(gamma, dtype=np.float32), (self.n_folds,)))
        c = _f32(np.broadcast_to(np.asarray(C, dtype=np.float32), (self.n_folds,)))
        it = np.zeros((self.n_folds, self.n_pairs), dtype=np.int32)
        self._chk(self.lib.mrgan_svm_fit_folds(self._h, _lib.iptr(lab), lab.shape[1], _lib.fptr(c), _lib.fptr(g), float(tol), _lib.iptr(it)))
        return it

    def svm_cv(self, lab_rows, split, C_grid, gamma, tol=1e-3):
        """The inner cross-validation of ``GridSearchCV(SVC(kernel='rbf'), {'C': C_grid, 'gamma': ...}, cv)`` for every fold:
        split: int [n_folds, n_lab], the inner split of each labeled row (0 .. n_splits - 1, n_splits = split.max() + 1);
        C_grid: [nC]; gamma: [n_folds, nG] (or [nG] for every fold), absolute.  Returns the misclassified validation rows,
        int32 [n_folds, nG, nC, n_splits].  Invalidates a previous svm_fit (svm_eval etc. fail until the next one)."""
        lab = self._svm_lab("svm_cv", lab_rows)
        sp = _i32(split)
        if sp.shape != lab.shape:
            raise ValueError("svm_cv: split must have the shape of lab_rows")
        c = _f32(np.atleast_1d(np.asarray(C_grid, dtype=np.float32)))
        g = np.asarray(gamma, dtype=np.float32)
        g = _f32(np.broadcast_to(g, (self.n_folds,) + g.shape[-1:]) if g.ndim == 1 else g)
        if g.ndim != 2 or g.shape[0] != self.n_folds:
            raise ValueError("svm_cv: gamma must be [nG] or [n_folds, nG]")
        ns = int(sp.max()) + 1 if sp.size else 0
        out = np.zeros((self.n_folds, g.shape[1], len(c), max(ns, 1)), dtype=np.int32)
        self._chk(self.lib.mrgan_svm_cv(self._h, _lib.iptr(lab), lab.shape[1], _lib.iptr(sp), ns, _lib.fptr(c), len(c), _lib.fptr(g),
                                        g.shape[1], float(tol), _lib.iptr(out)))
        return out

    def svm_eval(self, fold):
        """Error of the one-vs-one vote on the fold's full test set (np.mean(predicted != y_test))."""
        out = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.mrgan_svm_eval(self._h, int(fold), _lib.fptr(out)))
        return float(out[0])

    def svm_decision(self, fold):
        """Test hook: the one-vs-one decision values, float32 [n_test, n_pairs] (pairs (0,1), (0,2), ...)."""
        out = np.zeros((self.shapes[fold][2], self.n_pairs), dtype=np.float32)
        self._chk(self.lib.mrgan_svm_decision(self._h, int(fold), _lib.fptr(out)))
        return out

    # ------------------------------------------------------------------ predictions (all three models)
    def _n_scores(self):
        return self.n_pairs if self.model == "svm" else self.cfg.n_classes

    def predict(self, fold):
        """Predicted classes of the fold's resident test set and their raw scores: (int32 [n_test], float32 [n_test, K])
        logits (GAN / NN, phase 0) or (.., [n_test, n_pairs]) one-vs-one decision values (SVM)."""
        n = self.shapes[fold][2]
        pred = np.empty(n, dtype=np.int32)
        scores = np.empty((n, self._n_scores()), dtype=np.float32)
        self._chk(self.lib.mrgan_predict(self._h, int(fold), _lib.iptr(pred), _lib.fptr(scores)))
        return pred, scores

    def predict_rows(self, fold, x):
        """predict() for new rows x [n, D] in the fold's SCALED input space (that of the resident X_test), in chunks of at
        most n_test rows.  Leaves every later result on the resident test set unchanged."""
        D, _, nte, _ = self.shapes[fold]
        x = _f32(x)
        if x.ndim != 2 or x.shape[1] != D or x.shape[0] < 1:
            raise ValueError("predict_rows: x must be [n >= 1, %d]" % D)
        n = x.shape[0]
        pred = np.empty(n, dtype=np.int32)
        scores = np.empty((n, self._n_scores()), dtype=np.float32)
        for a in range(0, n, nte):
            b = min(n, a + nte)
            xc, pc, sc = x[a:b], pred[a:b], scores[a:b]       # contiguous row slices: the library writes straight into them
            self._chk(self.lib.mrgan_predict_rows(self._h, int(fold), _lib.fptr(xc), b - a, _lib.iptr(pc), _lib.fptr(sc)))
        return pred, scores

    def confusion(self):
        """Confusion counts of every fold's resident test set in one pass: int32 [n_folds, K, K], rows = true class,
        columns = predicted class."""
        K = self.cfg.n_classes
        out = np.zeros((self.n_folds, K, K), dtype=np.int32)
        self._chk(self.lib.mrgan_confusion(self._h, _lib.iptr(out)))
        return out

    # ------------------------------------------------------------------ input gradients (GAN / NN)
    def input_grad(self, fold, x=None, target=None):
        """d log softmax(l(x))[t] / dx of the fold's phase-0 logits l (those of predict), float32 [n, D], x in the fold's
        SCALED input space.  x: rows [n, D] (in chunks of at most n_test rows), or None = the resident X_test.  target: int
        [n] classes, or None = each row's predicted class.  Leaves every later result of the group unchanged."""
        D, _, nte, _ = self.shapes[fold]
        if x is None:
            n = nte
        else:
            x = _f32(x)
            if x.ndim != 2 or x.shape[1] != D or x.shape[0] < 1:
                raise ValueError("input_grad: x must be [n >= 1, %d]" % D)
            n = x.shape[0]
        if target is not None:
            target = _i32(target)
            if target.shape != (n,):
                raise ValueError("input_grad: target must be [%d]" % n)
        grad = np.empty((n, D), dtype=np.float32)
        for a in range(0, n, nte):
            b = min(n, a + nte)
            xp = None if x is None else _lib.fptr(x[a:b])
            tp = None if target is None else _lib.iptr(target[a:b])
            self._chk(self.lib.mrgan_input_grad(self._h, int(fold), xp, b - a, tp, _lib.fptr(grad[a:b])))
        return grad

    def saliency(self):
        """Saliency profile of every fold in one pass over its resident test set: a list of float32 [K, D_f], row c = the mean
        of |input_grad(f, target=y_test)| over the test rows of class c (zero for a class without test rows).  Bitwise
        reproducible and independent of the fold grouping."""
        K, Dmax = self.cfg.n_classes, max(s[0] for s in self.shapes)
        out = np.empty((self.n_folds, K, Dmax), dtype=np.float32)
        self._chk(self.lib.mrgan_saliency(self._h, _lib.fptr(out)))
        return [out[f, :, :D].copy() for f, (D, _, _, _) in enumerate(self.shapes)]

    # ------------------------------------------------------------------ utilities
    def fill_normal(self, fold, step, tensor_id, rows, cols, row0=0):
        out = np.empty((rows, cols), dtype=np.float32)
        self._chk(self.lib.mrgan_fill_normal(self._h, fold, step, tensor_id, rows, cols, row0, _lib.fptr(out)))
        return out

    def adam_flat(self, p, m, v, g, t):
        p, m, v, g = (_f32(a).copy() for a in (p, m, v, g))
        self._chk(self.lib.mrgan_adam_flat(self._h, _lib.fptr(p), _lib.fptr(m), _lib.fptr(v), _lib.fptr(g), p.size, t))
        return p, m, v

    def debug_buffer(self, fold, which, rows, cols):
        """Test hook: an intermediate buffer of the last step (see mrgan_debug_buffer in include/mrgan.h)."""
        out = np.empty((rows, cols), dtype=np.float32)
        self._chk(self.lib.mrgan_debug_buffer(self._h, fold, which, _lib.fptr(out), rows, cols))
        return out

    def debug_gemm(self, mode, A, B, use_tc=True):
        """Test hook: stand-alone GEMM through the step's kernels (see mrgan_debug_gemm)."""
        A, B = _f32(A), _f32(B)
        if mode == 0:
            M, K, N = A.shape[0], A.shape[1], B.shape[1]
        elif mode == 1:
            M, K, N = A.shape[0], A.shape[1], B.shape[0]
        else:
            K, M, N = A.shape[0], A.shape[1], B.shape[1]
        out = np.zeros((M, N), dtype=np.float32)
        self._chk(self.lib.mrgan_debug_gemm(self._h, mode, M, N, K, _lib.fptr(A), _lib.fptr(B), _lib.fptr(out), int(use_tc)))
        return out

    def debug_gemm_time(self, mode, M, N, K, groups=1, reps=20):
        out = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.mrgan_debug_gemm_time(self._h, mode, M, N, K, groups, reps, _lib.fptr(out)))
        return float(out[0])

    TIME_OPS = {"adam_d": 0, "adam_g": 1, "dw1": 2, "fwd1": 3, "disc_step": 4, "gen_step": 5, "dx1": 6,
                "svm_kmat": 7, "svm_smo": 8, "svm_predict": 9, "saliency": 10}

    def time_op(self, which, reps=20):
        """Average device ms of one kernel (or one whole step) over all folds; mutates training state (but 'saliency')."""
        out = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.mrgan_time_op(self._h, self.TIME_OPS[which], reps, _lib.fptr(out)))
        return float(out[0])

    @property
    def kernel_launches(self):
        return int(self.lib.mrgan_kernel_launches(self._h))

    @property
    def last_device_ms(self):
        return float(self.lib.mrgan_last_device_ms(self._h))
