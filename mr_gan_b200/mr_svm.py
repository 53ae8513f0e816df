"""Drop-in for the reference's ``mr_svm.py``: the RBF support vector machine baseline of tables 2 and 4
(``SVC(kernel='rbf', C=1.0)`` at mr_svm.py:106, per SURVEY.md row 7) and its ``--tables 2 4`` CLI (mr_svm.py:118-165),
on sm_100a kernels (csrc/kernels_svm.cuh): tcgen05 kernel matrices and a batched one-vs-one SMO solver that restates
sklearn's libsvm (sklearn/svm/src/libsvm/svm.cpp) without shrinking.

The reference's text is not reproduced here; SURVEY.md records mr_svm.py as the twin of mr_nn.py, so fold preparation,
seeding, printed strings and loop structure follow mr_nn.py's drop-in (mr_nn.py).  gamma defaults to 1 / D, the
``gamma='auto'`` default of the sklearn of the reference's stack.  The ``deriv`` feature option of mr_svm.py's copy
of ``dataset()`` is not supported.  There is no CPU fallback.

With ``grid`` (CLI: ``--tune``), every fold is instead ``GridSearchCV(SVC(kernel='rbf'), {'C': ..., 'gamma': ...},
cv=StratifiedKFold(cv))`` on its labeled rows, refit with the selected point: the inner fits run on the GPU
(``FoldGroup.svm_cv``), the scores and the choice are computed here exactly as sklearn computes them (``select``)."""
import argparse
import sys

import numpy as np
from sklearn.model_selection import StratifiedKFold

from . import foldprep, results, sweep
from .engine import FoldGroup
from .model import MATERIALS, fold_key
from .mr_gan import MODALITIES, _kfold_jobs, _loo_jobs, dataset, job_rows


def prepare_folds(jobs, seed):
    """Shuffled training rows and class-major labeled rows of every job, drawn exactly like mr_nn.train_nn_folds (the
    job's stream is seeded by (seed, job_id)), so that the SVM and NN columns of a table see the same folds."""
    folds = []
    for i, job in enumerate(jobs):
        rng = np.random.default_rng([int(seed), int(job.get('job_id', i))])
        if 'train_idx' in job:
            folds.append(foldprep.prepare_fold_indices(job['y'], job['train_idx'], job['test_idx'], job['percentlabeled'], None, rng))
        else:
            folds.append(foldprep.prepare_fold(job.get('X'), job.get('y'), job['percentlabeled'], None, job.get('trainTestSets'), rng))
    return folds


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
        errors = [fg.svm_eval(i) for i in range(len(jobs))]
        if details:
            errors = [dict(error=e, confusion=c) for e, c in zip(errors, fg.confusion())]
        if tuned is not None:
            errors = [dict(e if isinstance(e, dict) else dict(error=e), **t) for e, t in zip(errors, tuned)]
        return errors
    finally:
        fg.close()


def tune_group(jobs, grid, cv=5, verbose=False, *, seed=0, device=0):
    """Grid search of every fold of a group, then the refit with each fold's selected point.  Returns the fitted FoldGroup
    (the caller closes it) and per job ``{'C', 'gamma_D', 'cv_accuracy'}``."""
    Cs = [float(c) for c in grid['C']]
    gD = [float(g) for g in grid['gamma_D']]
    fg, folds, shapes = load_group(jobs, verbose, seed=seed, device=device)
    try:
        lab = np.stack([f.lab_rows for f in folds])
        split = np.stack([inner_splits(f.y_train[f.lab_rows], cv) for f in folds])
        D = np.array([s[0] for s in shapes], dtype=np.float64)
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
    fg, folds, shapes = load_group(jobs, verbose, seed=seed, device=device)
    try:
        gam = [1.0 / s[0] if gamma is None else float(gamma) for s in shapes]
        return fg, fg.svm_fit(np.stack([f.lab_rows for f in folds]), C=C, gamma=gam)
    except BaseException:
        fg.close()
        raise


def load_group(jobs, verbose=False, *, seed=0, device=0):
    """A FoldGroup (model='svm') holding the folds of a group of jobs, the jobs' prepared folds and their shapes."""
    folds = prepare_folds(jobs, seed)
    n_lab = len(folds[0].lab_rows)
    if any(len(f.lab_rows) != n_lab for f in folds):
        raise ValueError("folds of one group must have the same number of labeled rows")
    slots = {}
    for job in jobs:
        if 'train_idx' in job:
            slots.setdefault(id(job['X']), (len(slots), job['X'], job['y']))

    def dims(f, job):
        if isinstance(f, foldprep.FoldIndex):
            return job['X'].shape[1], len(f.train_rows), len(f.test_rows)
        return f.x_train.shape[1], f.x_train.shape[0], f.x_test.shape[0]

    shapes = [dims(f, job) + (fold_key(seed, job.get('job_id', i)),) for i, (f, job) in enumerate(zip(folds, jobs))]
    fg = FoldGroup(shapes, model='svm', device=device)
    try:
        for slot, X, y in slots.values():
            fg.load_dataset(slot, X, y)
        for i, (f, job) in enumerate(zip(folds, jobs)):
            D, ntr, nte = shapes[i][:3]
            if verbose:
                print('Num of class examples in test set:', [int(np.sum(f.y_test == c)) for c in range(len(MATERIALS))])
                print('X_train:', (ntr, D), 'y_train:', (ntr,), 'X_test:', (nte, D), 'y_test:', (nte,))
                print('x_labeled:', (n_lab, D), 'y_labeled:', (n_lab,))
            if isinstance(f, foldprep.FoldIndex):
                fg.prepare_fold(i, slots[id(job['X'])][0], f.train_rows, f.test_rows)
            else:
                fg.load_fold(i, f.x_train, f.y_train, f.x_test, f.y_test)
        return fg, folds, shapes
    except BaseException:
        fg.close()
        raise


def mr_svm(X, y, percentlabeled=50, trainTestSets=None, verbose=False, *, seed=None, device=0, C=1.0, gamma=None, grid=None, cv=5):
    """mr_svm.py:77-116, one fold; gamma=None means 1 / D.  With grid (see train_svm_folds) the fold is tuned by grid search
    and the result is a dict."""
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))      # mr_svm.py:78-79
    job = dict(X=X, y=y, percentlabeled=percentlabeled, trainTestSets=trainTestSets)
    return train_svm_folds([job], verbose=verbose, seed=seed, device=device, C=C, gamma=gamma, grid=grid, cv=cv)[0]


def selected_line(results):
    """The printed choice of a tuned setting's fold-trainings, in printed order."""
    return ('Selected C: ' + ' '.join('%g' % r['C'] for r in results) +
            ' Selected gamma*D: ' + ' '.join('%g' % r['gamma_D'] for r in results))


def table_jobs(tables, seed, data_dir='data_processed', synthetic=False):
    """(table, modality, percents, objects-or-None, jobs) of the sweep, in print order, with the job ids mr_nn.main gives."""
    out, jid = [], 0
    for t in ('2', '4'):
        if t not in tables:
            continue
        for modality in [2, 5]:
            if t == '2':
                X, y = dataset(modalities=modality, seed=seed, data_dir=data_dir, synthetic_data=synthetic)
                percents, objects = [1, 2, 4, 8, 16, 50, 100], None
                jobs = [j for p in percents for j in _kfold_jobs(X, y, seed + p, percentlabeled=p)]
            else:
                objects = dataset(modalities=modality, leaveObjectOut=True, seed=seed, data_dir=data_dir, synthetic_data=synthetic)
                percents = [1, 4, 16, 50, 100]
                jobs = [j for p in percents for j in _loo_jobs(objects, percentlabeled=p)]
            for j in jobs:
                j['job_id'] = jid
                jid += 1
            out.append((t, modality, percents, objects, jobs))
    return out


def main(argv=None):
    parser = argparse.ArgumentParser(description='Collecting data from a spinning platter of objects.')
    parser.add_argument('-t', '--tables', nargs='+', help='[Required] Tables to recompute', required=True)
    parser.add_argument('-v', '--verbose', help='Verbose', action='store_true')
    parser.add_argument('--seed', type=int, default=None)
    parser.add_argument('--group', type=int, default=42)
    parser.add_argument('--data-dir', default='data_processed')
    parser.add_argument('--synthetic', action='store_true', help='synthetic data of the MREO shape instead of the processed pickles')
    parser.add_argument('--tune', action='store_true',
                        help="tune C and gamma of every fold by grid search with stratified inner cross-validation (sklearn's "
                             "GridSearchCV) instead of the reference's C = 1, gamma = 1 / D")
    parser.add_argument('--C-grid', type=float, nargs='+', default=DEFAULT_GRID['C'], help='C values of --tune')
    parser.add_argument('--gamma-grid', type=float, nargs='+', default=DEFAULT_GRID['gamma_D'],
                        help='gamma values of --tune, as multiples of 1 / D')
    parser.add_argument('--cv', type=int, default=5, help='inner stratified splits of --tune')
    results.add_arguments(parser)
    args = parser.parse_args(argv)
    rank, world, local = sweep.dist_env()
    seed = sweep.shared_seed(args.seed)
    say = print if rank == 0 else (lambda *a, **k: None)
    if rank == 0:
        sys.stderr.write('seed: %d%s\n' % (seed, '   [SYNTHETIC data of the MREO shape: not the paper\'s dataset]' if args.synthetic else ''))
    rep = results.Report(args, 'mr_svm', rank, say, seed=seed)

    grid = dict(C=args.C_grid, gamma_D=args.gamma_grid) if args.tune else None
    work = 1 + len(args.C_grid) * len(args.gamma_grid) if args.tune else 1      # the fit, and one CV per grid point

    def run(jobs):
        return sweep.run_sharded(
            jobs, lambda js, dev: train_svm_folds(js, verbose=args.verbose, seed=seed, device=dev, details=rep.details, grid=grid,
                                                  cv=args.cv),
            group_size=args.group,
            key=lambda j: job_rows(j) + (j['percentlabeled'],),
            cost=lambda j: float(60 * j['percentlabeled']) ** 2 * work)   # n_lab^2: kernel matrix and SMO row traffic

    headed = set()
    for t, modality, percents, objects, jobs in table_jobs(args.tables, seed, args.data_dir, args.synthetic):
        if t not in headed:
            headed.add(t)
            if t == '2':
                say('\n', '-' * 25, 'Testing various amounts of labeled training data', '-' * 25)
            else:
                say('\n', '-' * 25, 'Testing generalization with leave-one-object-out validation', '-' * 25)
            say('-' * 100)
        say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)
        res = run(jobs)
        errors = results.errors(res)
        if t == '2':
            for k, p in enumerate(percents):
                say('-' * 15, 'Percentage of training data labeled: %d%%' % p, '-' * 15)
                e = errors[6 * k:6 * k + 6]
                say('Average error:', np.mean(e), 'Average accuracy:', np.mean(1.0 - np.array(e)))
                rep.setting(jobs[6 * k:6 * k + 6], res[6 * k:6 * k + 6], table=2, modality=MODALITIES[modality])
                if args.tune:
                    say(selected_line(res[6 * k:6 * k + 6]))
                sys.stdout.flush()
        else:
            n = len(objects)
            for k, p in enumerate(percents):
                say('-' * 15, 'Percentage of training data labeled: %d%%' % p, '-' * 15)
                for j, e in zip(jobs[n * k:n * k + n], errors[n * k:n * k + n]):
                    say(j['name'], 'Test error:', e, 'Test accuracy:', 1.0 - e)
                e = errors[n * k:n * k + n]
                say('Average leave-one-object-out error:', np.mean(e), 'Average accuracy:', np.mean(1.0 - np.array(e)))
                rep.setting(jobs[n * k:n * k + n], res[n * k:n * k + n], table=4, modality=MODALITIES[modality])
                if args.tune:
                    say(selected_line(res[n * k:n * k + n]))
                sys.stdout.flush()
    rep.close()
    return 0


if __name__ == '__main__':
    sys.exit(main())
