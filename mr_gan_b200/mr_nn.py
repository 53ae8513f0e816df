"""Drop-in for the reference's ``mr_nn.py``: the fully-supervised dense classifier (same
discriminator architecture, MSE vs one-hot, default Adam, batch 20; mr_nn.py:69-119) and its
``--tables 2 4`` CLI (mr_nn.py:121-168), on the same sm_100a kernels as the GAN path."""
import argparse
import sys

import numpy as np

from . import foldprep, results, sweep, synthetic
from .engine import FoldGroup
from .model import MATERIALS, fold_key, init_disc
from .mr_gan import MODALITIES, _kfold_jobs, _loo_jobs, dataset, job_rows, job_width


def train_nn_folds(jobs, epochs=100, verbose=False, *, seed=0, precision='f16', device=0, batch=20, details=False, saliency=False):
    """Train a group of independent mr_nn folds side by side; returns test errors (mr_nn.py:118-119), or with details=True
    one dict per job, ``{'error': <the same float>, 'confusion': int32 [K, K]}`` (rows = true class, columns = predicted);
    saliency=True: those dicts with ``'saliency'``, float32 [K, D] (FoldGroup.saliency)."""
    folds, rngs, slots = [], [], {}
    for i, job in enumerate(jobs):
        rng = np.random.default_rng([int(seed), int(job.get('job_id', i))])
        if 'train_idx' in job:
            folds.append(foldprep.prepare_fold_indices(job['y'], job['train_idx'], job['test_idx'], job['percentlabeled'], None, rng))
            slots.setdefault(id(job['X']), (len(slots), job['X'], job['y']))
        else:
            folds.append(foldprep.prepare_fold(job.get('X'), job.get('y'), job['percentlabeled'], None,
                                               job.get('trainTestSets'), rng))
        rngs.append(rng)
    n_lab = len(folds[0].lab_rows)
    if any(len(f.lab_rows) != n_lab for f in folds):
        raise ValueError("folds of one group must have the same number of labeled rows")
    if n_lab % batch:
        raise ValueError("labeled rows (%d) must be a multiple of the batch size (%d)" % (n_lab, batch))

    def dims(f, job):
        if isinstance(f, foldprep.FoldIndex):
            return job['X'].shape[1], len(f.train_rows), len(f.test_rows)
        return f.x_train.shape[1], f.x_train.shape[0], f.x_test.shape[0]

    shapes = [dims(f, job) + (fold_key(seed, job.get('job_id', i)),) for i, (f, job) in enumerate(zip(folds, jobs))]
    fg = FoldGroup(shapes, model='nn', precision=precision, device=device, batch=batch)
    for slot, X, y in slots.values():
        fg.load_dataset(slot, X, y)
    for i, (f, rng, job) in enumerate(zip(folds, rngs, jobs)):
        D, ntr, nte = shapes[i][:3]
        if verbose:
            print('Num of class examples in test set:', [int(np.sum(f.y_test == c)) for c in range(len(MATERIALS))])
            print('X_train:', (ntr, D), 'y_train:', (ntr,), 'X_test:', (nte, D), 'y_test:', (nte,))
            print('x_labeled:', (n_lab, D), 'y_labeled:', (n_lab,))
        fg.set_params(i, 0, init_disc(D, rng))
        if isinstance(f, foldprep.FoldIndex):
            fg.prepare_fold(i, slots[id(job['X'])][0], f.train_rows, f.test_rows)
        else:
            fg.load_fold(i, f.x_train, f.y_train, f.x_test, f.y_test)

    def draw():   # model.fit(shuffle=True): one permutation of the labeled rows per epoch (mr_nn.py:117)
        return np.stack([f.lab_rows[rng.permutation(n_lab)] for f, rng in zip(folds, rngs)]).astype(np.int32)

    nxt = draw()
    for epoch in range(epochs):
        fg.nn_train_epoch(nxt, wait=False)
        if epoch + 1 < epochs:
            nxt = draw()
    errors = [1.0 - float(fg.nn_evaluate(i)[1]) for i in range(len(jobs))]     # mr_nn.py:118
    if details or saliency:
        errors = [dict(error=e, confusion=c) for e, c in zip(errors, fg.confusion())]
    if saliency:
        for r, p in zip(errors, fg.saliency()):
            r['saliency'] = p
    fg.close()
    return errors


def mr_nn(X, y, percentlabeled=50, trainTestSets=None, verbose=False, *, seed=None, epochs=100, precision='f16',
          device=0):
    """mr_nn.py:69-119, one fold."""
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))      # mr_nn.py:70-71
    job = dict(X=X, y=y, percentlabeled=percentlabeled, trainTestSets=trainTestSets)
    return train_nn_folds([job], epochs=epochs, verbose=verbose, seed=seed, precision=precision, device=device)[0]


def main(argv=None):
    parser = argparse.ArgumentParser(description='Collecting data from a spinning platter of objects.')
    parser.add_argument('-t', '--tables', nargs='+', help='[Required] Tables to recompute', required=True)
    parser.add_argument('-v', '--verbose', help='Verbose', action='store_true')
    parser.add_argument('--seed', type=int, default=None)
    parser.add_argument('--epochs', type=int, default=100)
    parser.add_argument('--precision', choices=['fp32', 'tf32', 'f16'], default='f16',
                        help='arithmetic of the dense layers: f16 = fp16 operand copies, fp32 accumulation and master weights (default; per-step '
                             'losses within 1e-3 of the oracle, 43 k step-pairs/s per B200); tf32; fp32 = FFMA parity mode (1e-7, 9.8 k)')
    parser.add_argument('--group', type=int, default=42)
    parser.add_argument('--data-dir', default='data_processed')
    parser.add_argument('--synthetic', action='store_true', help='synthetic data of the MREO shape instead of the processed pickles')
    results.add_arguments(parser, saliency=True)
    args = parser.parse_args(argv)
    rank, world, local = sweep.dist_env()
    seed = sweep.shared_seed(args.seed)          # one seed for every rank: same dataset, same splits, same job streams
    say = print if rank == 0 else (lambda *a, **k: None)
    if rank == 0:
        sys.stderr.write('seed: %d%s\n' % (seed, '   [SYNTHETIC data of the MREO shape: not the paper\'s dataset]' if args.synthetic else ''))
    jid = [0]
    rep = results.Report(args, 'mr_nn', rank, say, seed=seed, precision=args.precision, epochs=args.epochs)

    def run(jobs):
        for j in jobs:
            j['job_id'] = jid[0]
            jid[0] += 1
        return sweep.run_sharded(
            jobs, lambda js, dev: train_nn_folds(js, epochs=args.epochs, verbose=args.verbose, seed=seed,
                                                 precision=args.precision, device=dev, details=rep.details,
                                                 saliency=rep.saliency),
            group_size=args.group,
            key=lambda j: job_rows(j) + (j['percentlabeled'],),
            cost=lambda j: job_width(j) * j['percentlabeled'])

    if '2' in args.tables:                      # mr_nn.py:129-146
        say('\n', '-' * 25, 'Testing various amounts of labeled training data', '-' * 25)
        say('-' * 100)
        for modality in [2, 5]:
            say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)
            X, y = dataset(modalities=modality, seed=seed, data_dir=args.data_dir, synthetic_data=args.synthetic)
            percents = [1, 2, 4, 8, 16, 50, 100]
            jobs = [j for p in percents for j in _kfold_jobs(X, y, seed + p, percentlabeled=p)]
            res = run(jobs)
            errors = results.errors(res)
            for k, p in enumerate(percents):
                say('-' * 15, 'Percentage of training data labeled: %d%%' % p, '-' * 15)
                e = errors[6 * k:6 * k + 6]
                say('Average error:', np.mean(e), 'Average accuracy:', np.mean(1.0 - np.array(e)))
                rep.setting(jobs[6 * k:6 * k + 6], res[6 * k:6 * k + 6], synthetic.block_widths(modality), table=2,
                            modality=MODALITIES[modality])
                sys.stdout.flush()

    if '4' in args.tables:                      # mr_nn.py:148-168
        say('\n', '-' * 25, 'Testing generalization with leave-one-object-out validation', '-' * 25)
        say('-' * 100)
        for modality in [2, 5]:
            say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)
            objects = dataset(modalities=modality, leaveObjectOut=True, seed=seed, data_dir=args.data_dir, synthetic_data=args.synthetic)
            percents = [1, 4, 16, 50, 100]
            jobs = [j for p in percents for j in _loo_jobs(objects, percentlabeled=p)]
            res = run(jobs)
            errors = results.errors(res)
            n = len(objects)
            for k, p in enumerate(percents):
                say('-' * 15, 'Percentage of training data labeled: %d%%' % p, '-' * 15)
                for j, e in zip(jobs[n * k:n * k + n], errors[n * k:n * k + n]):
                    say(j['name'], 'Test error:', e, 'Test accuracy:', 1.0 - e)
                e = errors[n * k:n * k + n]
                say('Average leave-one-object-out error:', np.mean(e), 'Average accuracy:', np.mean(1.0 - np.array(e)))
                rep.setting(jobs[n * k:n * k + n], res[n * k:n * k + n], synthetic.block_widths(modality), table=4,
                            modality=MODALITIES[modality])
                sys.stdout.flush()
    rep.close()
    return 0


if __name__ == '__main__':
    sys.exit(main())
