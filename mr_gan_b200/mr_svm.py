"""Drop-in for the reference's ``mr_svm.py``: the RBF support vector machine baseline of tables 2 and 4
(``SVC(kernel='rbf', C=1.0)`` at mr_svm.py:106, per SURVEY.md row 7) and its ``--tables 2 4`` CLI (mr_svm.py:118-165),
on sm_100a kernels (csrc/kernels_svm.cuh): tcgen05 kernel matrices and a batched one-vs-one SMO solver that restates
sklearn's libsvm (sklearn/svm/src/libsvm/svm.cpp) without shrinking.

The reference's text is not reproduced here; SURVEY.md records mr_svm.py as the twin of mr_nn.py, so fold preparation,
seeding, printed strings and loop structure follow mr_nn.py's drop-in (mr_nn.py).  gamma defaults to 1 / D, the
``gamma='auto'`` default of the sklearn of the reference's stack.  The ``deriv`` feature option of mr_svm.py's copy
of ``dataset()`` is not supported.  There is no CPU fallback."""
import argparse
import sys

import numpy as np

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


def train_svm_folds(jobs, verbose=False, *, seed=0, device=0, C=1.0, gamma=None, details=False):
    """Fit a group of independent mr_svm folds side by side; returns their test errors, or with details=True one dict per
    job, ``{'error': <the same float>, 'confusion': int32 [K, K]}`` (rows = true class, columns = predicted)."""
    fg, _ = fit_group(jobs, verbose, seed=seed, device=device, C=C, gamma=gamma)
    try:
        errors = [fg.svm_eval(i) for i in range(len(jobs))]
        if details:
            errors = [dict(error=e, confusion=c) for e, c in zip(errors, fg.confusion())]
        return errors
    finally:
        fg.close()


def fit_group(jobs, verbose=False, *, seed=0, device=0, C=1.0, gamma=None):
    """The fitted FoldGroup of a group of jobs (the caller closes it) and the SMO iterations [n_folds, n_pairs]."""
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
        gam = [1.0 / s[0] if gamma is None else float(gamma) for s in shapes]
        return fg, fg.svm_fit(np.stack([f.lab_rows for f in folds]), C=C, gamma=gam)
    except BaseException:
        fg.close()
        raise


def mr_svm(X, y, percentlabeled=50, trainTestSets=None, verbose=False, *, seed=None, device=0, C=1.0, gamma=None):
    """mr_svm.py:77-116, one fold; gamma=None means 1 / D."""
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))      # mr_svm.py:78-79
    job = dict(X=X, y=y, percentlabeled=percentlabeled, trainTestSets=trainTestSets)
    return train_svm_folds([job], verbose=verbose, seed=seed, device=device, C=C, gamma=gamma)[0]


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
    results.add_arguments(parser)
    args = parser.parse_args(argv)
    rank, world, local = sweep.dist_env()
    seed = sweep.shared_seed(args.seed)
    say = print if rank == 0 else (lambda *a, **k: None)
    if rank == 0:
        sys.stderr.write('seed: %d%s\n' % (seed, '   [SYNTHETIC data of the MREO shape: not the paper\'s dataset]' if args.synthetic else ''))
    rep = results.Report(args, 'mr_svm', rank, say, seed=seed)

    def run(jobs):
        return sweep.run_sharded(
            jobs, lambda js, dev: train_svm_folds(js, verbose=args.verbose, seed=seed, device=dev, details=rep.details),
            group_size=args.group,
            key=lambda j: job_rows(j) + (j['percentlabeled'],),
            cost=lambda j: float(60 * j['percentlabeled']) ** 2)          # n_lab^2: kernel matrix and SMO row traffic

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
                sys.stdout.flush()
    rep.close()
    return 0


if __name__ == '__main__':
    sys.exit(main())
