"""Drop-in for the reference's ``mr_svm.py``: the RBF support vector machine baseline of tables 2 and 4
(``SVC(kernel='rbf', C=1.0)`` at mr_svm.py:106, per SURVEY.md row 7) and its ``--tables 2 4`` CLI (mr_svm.py:118-165),
on sm_100a kernels (csrc/kernels_svm.cuh): tcgen05 kernel matrices and a batched one-vs-one SMO solver that restates
sklearn's libsvm (sklearn/svm/src/libsvm/svm.cpp) without shrinking.

The reference's text is not reproduced here; SURVEY.md records mr_svm.py as the twin of mr_nn.py, so fold preparation and
seeding (foldprep.load_folds), printed strings and the tables' jobs (tables.py) are mr_nn.py's drop-in's.  gamma defaults to 1 / D, the
``gamma='auto'`` default of the sklearn of the reference's stack.  The ``deriv`` feature option of mr_svm.py's copy
of ``dataset()`` is not supported.  There is no CPU fallback.

With ``grid`` (CLI: ``--tune``), every fold is instead ``GridSearchCV(SVC(kernel='rbf'), {'C': ..., 'gamma': ...},
cv=StratifiedKFold(cv))`` on its labeled rows, refit with the selected point: the inner fits run on the GPU
(``FoldGroup.svm_cv``), the scores and the choice are computed here exactly as sklearn computes them (``select``)."""
import sys

import numpy as np
from sklearn.model_selection import StratifiedKFold

from . import foldprep, results, tables
from .engine import FoldGroup
from .tables import job_rows


# The tuning grid of --tune: C absolute, gamma as a multiple of 1 / D (one grid for the mixed widths of a group).  It holds
# the reference's point (C = 1, gamma = 1 / D).
DEFAULT_GRID = {'C': [0.1, 1, 10, 100], 'gamma_D': [0.25, 0.5, 1, 2, 4]}


def inner_splits(y_lab, n_splits):
    """The inner split (0 .. n_splits - 1) of every labeled row: the validation folds of sklearn's
    ``StratifiedKFold(n_splits)`` without shuffling, which ``GridSearchCV(cv=n_splits)`` uses for a classifier."""
    y = np.asarray(y_lab)
    counts = np.unique(y, return_counts=True)[1]
    if n_splits > counts.min():
        raise ValueError("n_splits=%d is larger than the smallest class count %d of the labeled rows" % (n_splits, counts.min()))
    split = np.empty(len(y), np.int32)
    for s, (_, val) in enumerate(StratifiedKFold(n_splits).split(np.zeros((len(y), 1)), y)):
        split[val] = s
    return split


def select(wrong, n_val):
    """GridSearchCV's scores and choice for one fold.  wrong: int [nG, nC, n_splits] misclassified validation rows (the
    layout of FoldGroup.svm_cv); n_val: int [n_splits] validation rows.  Returns (mean, (iC, iG)): mean = float64 [nC, nG],
    sklearn's mean_test_score in ParameterGrid order (keys sorted: C outer, gamma inner), and the first point with the
    largest mean (sklearn's rankdata(-mean, 'min').argmin())."""
    w = np.asarray(wrong, dtype=np.int64).transpose(1, 0, 2)
    n = np.asarray(n_val, dtype=np.int64)
    acc = (n - w) / n                         # accuracy_score: the mean of exact 0 / 1 values, one correctly rounded division
    nC, nG, ns = acc.shape
    mean = np.average(np.array(acc, dtype=np.float64).reshape(nC * nG, ns), axis=1)   # BaseSearchCV._format_results
    best = int(np.argmax(mean))               # the first maximum: rankdata(-mean, 'min').argmin()
    return mean.reshape(nC, nG), divmod(best, nG)


def train_svm_folds(jobs, verbose=False, *, seed=0, device=0, C=1.0, gamma=None, details=False, grid=None, cv=5):
    """Fit a group of independent mr_svm folds side by side; returns their test errors, or with details=True one dict per
    job, ``{'error': <the same float>, 'confusion': int32 [K, K]}`` (rows = true class, columns = predicted).
    grid = {'C': [...], 'gamma_D': [...]} tunes every fold by grid search with ``cv`` stratified inner splits instead of
    using C and gamma; the results are then dicts that also hold the selected ``'C'`` and ``'gamma_D'`` (gamma * D) and
    ``'cv_accuracy'``, float64 [nC, nG] mean inner accuracies."""
    if grid is None:
        fg, _ = fit_group(jobs, verbose, seed=seed, device=device, C=C, gamma=gamma)
        tuned = None
    else:
        fg, tuned = tune_group(jobs, grid, cv, verbose, seed=seed, device=device)
    try:
        return results.collect(fg, [fg.svm_eval(i) for i in range(len(jobs))], details, extra=tuned)
    finally:
        fg.close()


def tune_group(jobs, grid, cv=5, verbose=False, *, seed=0, device=0):
    """Grid search of every fold of a group, then the refit with each fold's selected point.  Returns the fitted FoldGroup
    (the caller closes it) and per job ``{'C', 'gamma_D', 'cv_accuracy'}``."""
    Cs = [float(c) for c in grid['C']]
    gD = [float(g) for g in grid['gamma_D']]
    fg, folds = load_group(jobs, verbose, seed=seed, device=device)
    try:
        lab = np.stack([f.lab_rows for f in folds])
        split = np.stack([inner_splits(f.y_train[f.lab_rows], cv) for f in folds])
        D = np.array([s[0] for s in fg.shapes], dtype=np.float64)
        wrong = fg.svm_cv(lab, split, Cs, np.array(gD)[None, :] / D[:, None])
        out = []
        for w, sp in zip(wrong, split):
            mean, (ic, ig) = select(w, np.bincount(sp, minlength=cv))
            out.append(dict(C=Cs[ic], gamma_D=gD[ig], cv_accuracy=mean))
        fg.svm_fit(lab, C=[t['C'] for t in out], gamma=[t['gamma_D'] / d for t, d in zip(out, D)])
        return fg, out
    except BaseException:
        fg.close()
        raise


def fit_group(jobs, verbose=False, *, seed=0, device=0, C=1.0, gamma=None):
    """The fitted FoldGroup of a group of jobs (the caller closes it) and the SMO iterations [n_folds, n_pairs]."""
    fg, folds = load_group(jobs, verbose, seed=seed, device=device)
    try:
        gam = [1.0 / s[0] if gamma is None else float(gamma) for s in fg.shapes]
        return fg, fg.svm_fit(np.stack([f.lab_rows for f in folds]), C=C, gamma=gam)
    except BaseException:
        fg.close()
        raise


def prepare_folds(jobs, seed):
    """The jobs' folds as the SVM (and the NN) draws them: the shuffled training rows and class-major labeled rows."""
    return foldprep.prepare_folds(jobs, seed)[0]


def load_group(jobs, verbose=False, *, seed=0, device=0):
    """A FoldGroup (model='svm') holding the folds of a group of jobs (the caller closes it), and the jobs' folds."""
    fg, folds, _ = foldprep.load_folds(jobs, seed, lambda shapes: FoldGroup(shapes, model='svm', device=device), verbose=verbose,
                                       same_labeled=True)
    return fg, folds


def mr_svm(X, y, percentlabeled=50, trainTestSets=None, verbose=False, *, seed=None, device=0, C=1.0, gamma=None, grid=None, cv=5):
    """mr_svm.py:77-116, one fold; gamma=None means 1 / D.  With grid (see train_svm_folds) the fold is tuned by grid search
    and the result is a dict."""
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))      # mr_svm.py:78-79
    job = dict(X=X, y=y, percentlabeled=percentlabeled, trainTestSets=trainTestSets)
    return train_svm_folds([job], verbose=verbose, seed=seed, device=device, C=C, gamma=gamma, grid=grid, cv=cv)[0]


def main(argv=None):
    parser = tables.argument_parser('Collecting data from a spinning platter of objects.', group=42, nets=False)
    parser.add_argument('--tune', action='store_true',
                        help="tune C and gamma of every fold by grid search with stratified inner cross-validation (sklearn's "
                             "GridSearchCV) instead of the reference's C = 1, gamma = 1 / D")
    parser.add_argument('--C-grid', type=float, nargs='+', default=DEFAULT_GRID['C'], help='C values of --tune')
    parser.add_argument('--gamma-grid', type=float, nargs='+', default=DEFAULT_GRID['gamma_D'],
                        help='gamma values of --tune, as multiples of 1 / D')
    parser.add_argument('--cv', type=int, default=5, help='inner stratified splits of --tune')
    args = parser.parse_args(argv)
    grid = dict(C=args.C_grid, gamma_D=args.gamma_grid) if args.tune else None
    work = 1 + len(args.C_grid) * len(args.gamma_grid) if args.tune else 1      # the fit, and one CV per grid point

    def train(jobs, device, seed, rep):
        return train_svm_folds(jobs, verbose=args.verbose, seed=seed, device=device, details=rep.details, grid=grid, cv=args.cv)

    return tables.run(args, 'mr_svm', train, lambda j: job_rows(j) + (j['percentlabeled'],),
                      lambda j: float(60 * j['percentlabeled']) ** 2 * work, ['2', '4'])   # n_lab^2: kernel matrix and SMO row traffic


if __name__ == '__main__':
    sys.exit(main())
