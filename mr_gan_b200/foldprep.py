"""Host-side fold preparation and epoch permutations of the reference, seedable.

mr_gan.py:86-107 (split, StandardScaler, shuffle, labeled / unlabeled subsets) and
mr_gan.py:189-202 (tiled permutations).  The reference uses numpy's unseeded global RNG
(mr_gan.py:74-75); here every draw comes from an explicit ``numpy.random.Generator`` so runs
are reproducible.  The device receives ROW INDICES into the resident X_train instead of the
gathered copies the reference builds every epoch (SURVEY.md a13).  ``load_folds`` prepares and loads the folds of a
group of jobs for all three trainers (GAN, NN, SVM)."""
from collections import namedtuple

import numpy as np
from sklearn import preprocessing
from sklearn.model_selection import train_test_split

from .model import MATERIALS, fold_key

FoldData = namedtuple("FoldData", "x_train y_train x_test y_test lab_rows unl_rows")


def prepare_fold(X, y, percentlabeled, percentunlabeled=None, trainTestSets=None, rng=None, n_classes=6):
    rng = rng if rng is not None else np.random.default_rng()
    test_ratio = 200 * n_classes                                  # mr_gan.py:81
    if trainTestSets is None:                                     # mr_gan.py:87-88
        X_train, X_test, y_train, y_test = train_test_split(
            X, y, test_size=test_ratio, stratify=y, random_state=int(rng.integers(2 ** 31)))
    else:
        X_train, X_test, y_train, y_test = trainTestSets          # mr_gan.py:90
    scaler = preprocessing.StandardScaler()                       # mr_gan.py:96-98
    X_train = scaler.fit_transform(np.asarray(X_train, dtype=np.float64))
    X_test = scaler.transform(np.asarray(X_test, dtype=np.float64))
    y_train, y_test = np.asarray(y_train), np.asarray(y_test)
    perm = rng.permutation(len(X_train))                          # sklearn.utils.shuffle, mr_gan.py:101
    X_train, y_train = X_train[perm], y_train[perm]
    lab_rows, unl_rows = _subsets(y_train, percentlabeled, percentunlabeled, n_classes)
    return FoldData(X_train.astype(np.float32), y_train.astype(np.int32), X_test.astype(np.float32),
                    y_test.astype(np.int32), lab_rows, unl_rows)


def _subsets(y_train, percentlabeled, percentunlabeled, n_classes):
    """Rows of the shuffled training set: the labeled ones, the first 10 x percentlabeled of every class (mr_gan.py:82,102),
    and with percentunlabeled the unlabeled pool, the first 10 x (percentlabeled + percentunlabeled) (mr_gan.py:106-107).
    Draws nothing."""
    def first(n):
        return np.concatenate([np.nonzero(y_train == j)[0][:n] for j in range(n_classes)])
    num_labeled = int(10 * percentlabeled)
    return first(num_labeled), None if percentunlabeled is None else first(num_labeled + int(10 * percentunlabeled))


def tiled_perm(rng, n_total, n_sub):
    """mr_gan.py:189: floor(N/L) permutations of L rows followed by a permutation of N mod L."""
    parts = [rng.permutation(n_sub) for _ in range(n_total // n_sub)]
    parts.append(rng.permutation(n_total % n_sub))
    return np.concatenate(parts).astype(np.int64)


def epoch_indices(rng, n_train, lab_rows, unl_rows=None):
    """Row indices into X_train of trainx / trainx_unl / trainx_unl2 (mr_gan.py:189-202).

    The third unlabeled permutation the reference draws and never uses (trainx_unl3) is drawn
    and discarded so the generator advances exactly as the reference's does."""
    idx_lab = lab_rows[tiled_perm(rng, n_train, len(lab_rows))]
    if unl_rows is None:
        u1, u2, _ = (rng.permutation(n_train) for _ in range(3))
    else:
        u1, u2, _ = (unl_rows[tiled_perm(rng, n_train, len(unl_rows))] for _ in range(3))
    return idx_lab.astype(np.int32), np.asarray(u1, np.int32), np.asarray(u2, np.int32)


FoldIndex = namedtuple("FoldIndex", "train_rows test_rows y_train y_test lab_rows unl_rows")


def prepare_fold_indices(y, train_idx, test_idx, percentlabeled, percentunlabeled=None, rng=None, n_classes=6):
    """Index-only version of ``prepare_fold`` for the device-side fold preparation (``FoldGroup.prepare_fold``):
    the same shuffle and labeled / unlabeled subset selection (mr_gan.py:101-107), but X never leaves the GPU.
    Draws from ``rng`` exactly like ``prepare_fold(trainTestSets=...)`` does, so both paths pick identical rows."""
    rng = rng if rng is not None else np.random.default_rng()
    y = np.asarray(y)
    train_idx, test_idx = np.asarray(train_idx), np.asarray(test_idx)
    perm = rng.permutation(len(train_idx))
    train_rows = train_idx[perm]
    y_train = y[train_rows]
    lab_rows, unl_rows = _subsets(y_train, percentlabeled, percentunlabeled, n_classes)
    return FoldIndex(train_rows.astype(np.int32), test_idx.astype(np.int32), y_train.astype(np.int32),
                     y[test_idx].astype(np.int32), lab_rows, unl_rows)


def prepare_folds(jobs, seed):
    """The fold of every job, drawn first from the job's own stream ``default_rng([seed, job_id])`` (job_id: the job's
    index when it has none), and the streams, which the trainers go on drawing weights and permutations from.  A job is
    ``{'X', 'y', 'train_idx', 'test_idx'}`` (an index job, cut on the device by ``prepare_fold_indices``) or
    ``{'trainTestSets'}`` / ``{'X', 'y'}`` (``prepare_fold``), with ``percentlabeled`` and optionally ``percentunlabeled``."""
    rngs = [np.random.default_rng([int(seed), int(job.get('job_id', i))]) for i, job in enumerate(jobs)]
    folds = [prepare_fold_indices(job['y'], job['train_idx'], job['test_idx'], job['percentlabeled'], job.get('percentunlabeled'), rng)
             if 'train_idx' in job else
             prepare_fold(job.get('X'), job.get('y'), job['percentlabeled'], job.get('percentunlabeled'), job.get('trainTestSets'), rng)
             for job, rng in zip(jobs, rngs)]
    return folds, rngs


def load_folds(jobs, seed, make_group, init=None, verbose=False, same_labeled=False):
    """A fold group holding the prepared folds of jobs (prepare_folds): make_group(shapes) creates it from the folds'
    (D, n_train, n_test, fold key); every dataset the index jobs share is uploaded once; then per fold init(fg, i, D, rng)
    sets the initial weights from the fold's stream and the fold is loaded.  same_labeled: every fold must have as many
    labeled rows as the others (the NN and SVM train them as one block).  Returns (group, folds, streams); the group is
    closed if loading fails."""
    folds, rngs = prepare_folds(jobs, seed)
    slots = {}
    for job in jobs:
        if 'train_idx' in job:
            slots.setdefault(id(job['X']), (len(slots), job['X'], job['y']))
    if len(slots) > 8:
        raise ValueError("a fold group may draw from at most 8 datasets")
    if same_labeled and any(len(f.lab_rows) != len(folds[0].lab_rows) for f in folds):
        raise ValueError("folds of one group must have the same number of labeled rows")
    shapes = [(job['X'].shape[1], len(f.train_rows), len(f.test_rows)) if isinstance(f, FoldIndex) else
              (f.x_train.shape[1], f.x_train.shape[0], f.x_test.shape[0]) for f, job in zip(folds, jobs)]
    fg = make_group([s + (fold_key(seed, job.get('job_id', i)),) for i, (s, job) in enumerate(zip(shapes, jobs))])
    try:
        for slot, X, y in slots.values():
            fg.load_dataset(slot, X, y)            # one upload per dataset; every fold of the group reuses it
        for i, (f, rng, job, (D, ntr, nte)) in enumerate(zip(folds, rngs, jobs, shapes)):
            if verbose:
                print('Num of class examples in test set:', [int(np.sum(f.y_test == c)) for c in range(len(MATERIALS))])
                print('X_train:', (ntr, D), 'y_train:', (ntr,), 'X_test:', (nte, D), 'y_test:', (nte,))
                print('x_labeled:', (len(f.lab_rows), D), 'y_labeled:', (len(f.lab_rows),))
            if init is not None:
                init(fg, i, D, rng)
            if isinstance(f, FoldIndex):
                fg.prepare_fold(i, slots[id(job['X'])][0], f.train_rows, f.test_rows)
            else:
                fg.load_fold(i, f.x_train, f.y_train, f.x_test, f.y_test)
        return fg, folds, rngs
    except BaseException:
        fg.close()
        raise
