"""Drop-in for the reference's ``mr_gan.py``: same ``dataset()`` / ``mr_gan()`` signatures,
same ``--tables`` CLI and stdout strings (mr_gan.py:236-341), with the compiled training step
(mr_gan.py:169-171) and the epoch loop (mr_gan.py:183-230) running as sm_100a CUDA behind the
C-ABI of include/mrgan.h.  New arguments are keyword-only and default to the reference's
behaviour.  No CPU fallback: without a B200 ``mr_gan()`` raises."""
import argparse
import os
import sys
import time

import numpy as np
from sklearn.model_selection import StratifiedKFold

from . import foldprep, results, sweep, synthetic
from .engine import FoldGroup
from .model import MATERIALS, fold_key, init_disc, init_gen

MODALITIES = ['Force', 'Temperature', 'Force and Temperature', 'Contact mic', 'Temperature and Contact Mic',
              'Force, Temperature, and Contact Mic', 'Force and Contact Mic']      # mr_gan.py:237


def dataset(modalities=0, forcetempTime=4, contactmicTime=0.2, leaveObjectOut=False, verbose=False, *,
            seed=0, data_dir='data_processed', synthetic_data=False):
    """mr_gan.py:23-71.  Loads the processed MREO pickles from ``data_dir`` and, like the reference, raises IOError when
    they are missing.  The pickles are not distributed with the reference, so data of the same shape can be
    synthesised instead (synthetic.py) -- only on request (``synthetic_data=True`` / ``--synthetic``): a mistyped path
    must not silently turn into plausible-looking numbers."""
    if not synthetic_data:
        path = os.path.join(data_dir, 'processed_0.1sbefore_%s_times_%.2f_%.2f.pkl' % (MATERIALS[0], forcetempTime, contactmicTime))
        if not os.path.exists(path):
            raise IOError("processed MREO data not found: %s (pass synthetic_data=True / --synthetic for synthetic data "
                          "of the MREO shape)" % path)
        from .realdata import load_processed
        return load_processed(modalities, forcetempTime, contactmicTime, leaveObjectOut, verbose, data_dir)
    out = synthetic.synthetic_dataset(modalities, forcetempTime, contactmicTime, leaveObjectOut, seed=seed)
    if verbose and not leaveObjectOut:
        print('X:', np.shape(out[0]), 'y:', np.shape(out[1]), '(synthetic MREO shape)')
    return out


def train_gan_folds(jobs, epochs=100, verbose=False, *, seed=0, precision='f16', device=0, batch=50,
                    eval_each_epoch=True, shared_t=True, return_group=False, device_perm=False, details=False, saliency=False):
    """Train a GROUP of independent folds side by side on one GPU.

    jobs: list of dicts with keys ``trainTestSets`` (or ``X``, ``y``), ``percentlabeled``,
    ``percentunlabeled`` (optional), ``job_id`` (optional, seeds the fold's streams).
    device_perm: draw the epoch permutations of mr_gan.py:189-202 on the device (the host then sends one epoch number per
    epoch instead of 3 x int32[n_train] per fold); same distribution, different draws than the host's numpy generator.
    Returns the list of test errors (mr_gan.py:230,234), one per job; details=True: one dict per job instead,
    ``{'error': <the same float>, 'confusion': int32 [K, K]}`` (rows = true class, columns = predicted), from one extra
    forward pass over every fold's test set; saliency=True: those dicts with ``'saliency'``, float32 [K, D] (FoldGroup.saliency)."""
    folds, rngs, slots = [], [], {}
    for i, job in enumerate(jobs):
        rng = np.random.default_rng([int(seed), int(job.get('job_id', i))])
        if 'train_idx' in job:      # index job: the fold is cut on the device from the resident dataset
            folds.append(foldprep.prepare_fold_indices(job['y'], job['train_idx'], job['test_idx'], job['percentlabeled'],
                                                       job.get('percentunlabeled'), rng))
            slots.setdefault(id(job['X']), (len(slots), job['X'], job['y']))
        else:
            folds.append(foldprep.prepare_fold(job.get('X'), job.get('y'), job['percentlabeled'],
                                               job.get('percentunlabeled'), job.get('trainTestSets'), rng))
        rngs.append(rng)
    if len(slots) > 8:
        raise ValueError("a fold group may draw from at most 8 datasets")

    def dims(f, job):
        if isinstance(f, foldprep.FoldIndex):
            return job['X'].shape[1], len(f.train_rows), len(f.test_rows)
        return f.x_train.shape[1], f.x_train.shape[0], f.x_test.shape[0]

    shapes = [dims(f, job) + (fold_key(seed, job.get('job_id', i)),) for i, (f, job) in enumerate(zip(folds, jobs))]
    fg = FoldGroup(shapes, model='gan', precision=precision, device=device, batch=batch,
                   eval_each_epoch=eval_each_epoch, shared_t=shared_t)
    for slot, X, y in slots.values():
        fg.load_dataset(slot, X, y)            # one upload per dataset; every fold of the group reuses it
    for i, (f, rng, job) in enumerate(zip(folds, rngs, jobs)):
        D, ntr, nte = shapes[i][:3]
        if verbose:
            print('Num of class examples in test set:', [int(np.sum(f.y_test == c)) for c in range(len(MATERIALS))])
            print('X_train:', (ntr, D), 'y_train:', (ntr,), 'X_test:', (nte, D), 'y_test:', (nte,))
            print('x_labeled:', (len(f.lab_rows), D), 'y_labeled:', (len(f.lab_rows),))
        fg.set_params(i, 1, init_gen(D, rng))       # generator first, as mr_gan.py:110-114 builds it first
        fg.set_params(i, 0, init_disc(D, rng))
        if isinstance(f, foldprep.FoldIndex):
            fg.prepare_fold(i, slots[id(job['X'])][0], f.train_rows, f.test_rows)
        else:
            fg.load_fold(i, f.x_train, f.y_train, f.x_test, f.y_test)
    n_train = shapes[0][1]
    if verbose:
        print('Epochs:', epochs)
        print('Batch size:', batch)
        print('Training batches per epoch:', n_train // batch)
        print('Testing batches per epoch:', shapes[0][2] // batch)

    def draw():
        per = [foldprep.epoch_indices(rng, n_train, f.lab_rows, f.unl_rows) for f, rng in zip(folds, rngs)]
        return [np.stack([p[s] for p in per]) for s in range(3)]

    if device_perm and max(len(f.lab_rows) for f in folds) <= 8192 and all(
            (len(f.unl_rows) if f.unl_rows is not None else n_train) <= 8192 for f in folds):
        for i, f in enumerate(folds):
            fg.set_epoch_rows(i, f.lab_rows, f.unl_rows)
    else:
        device_perm = False
    nxt = None if device_perm else draw()
    for epoch in range(1, epochs + 1):
        begin = time.time()
        if device_perm:
            fg.train_epoch_seeded(epoch, wait=False)  # permutations drawn on the device from (fold key, epoch)
        else:
            fg.train_epoch(*nxt, wait=False)      # one CUDA-graph launch: the whole epoch, all folds
            if epoch < epochs:
                nxt = draw()                      # host permutations of the next epoch overlap the GPU
        st = fg.epoch_result()
        if verbose:
            for i in range(len(jobs)):
                print('Epoch %d, time = %ds, loss labeled = %.4f, loss unlabeled = %.4f, train error = %.4f, test error = %.4f'
                      % (epoch, time.time() - begin, st[i, 0], st[i, 1], st[i, 2], st[i, 4]))
            sys.stdout.flush()
    errors = [float(fg.eval(i)) for i in range(len(jobs))]
    if verbose:
        for e in errors:
            print('Test error:', e)
        sys.stdout.flush()
    if details or saliency:
        errors = [dict(error=e, confusion=c) for e, c in zip(errors, fg.confusion())]
    if saliency:
        for r, p in zip(errors, fg.saliency()):
            r['saliency'] = p
    if return_group:
        return errors, fg
    fg.close()
    return errors


def mr_gan(X, y, percentlabeled=50, percentunlabeled=None, epochs=100, trainTestSets=None, verbose=False, *,
           seed=None, precision='f16', device=0, batch=50, device_perm=False):
    """mr_gan.py:73-234, one fold.  ``seed=None`` reproduces the reference's 'Non Deterministic output'."""
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))      # mr_gan.py:74-75
    job = dict(X=X, y=y, percentlabeled=percentlabeled, percentunlabeled=percentunlabeled, trainTestSets=trainTestSets)
    return train_gan_folds([job], epochs=epochs, verbose=verbose, seed=seed, precision=precision, device=device,
                           batch=batch, device_perm=device_perm)[0]


# ------------------------------------------------------------------ CLI (mr_gan.py:236-341)
def _kfold_jobs(X, y, seed, **kw):
    """mr_gan.py:255-257 as index jobs: the split is expressed as row indices into the shared X."""
    skf = StratifiedKFold(n_splits=6, shuffle=True, random_state=seed)            # mr_gan.py:255
    return [dict(X=X, y=y, train_idx=tr, test_idx=te, **kw) for tr, te in skf.split(X, y)]


def stack_objects(objects):
    """Leave-one-object-out data as one matrix + per-object row ranges (mr_gan.py:274-278 concatenates per fold)."""
    names = list(objects)
    X = np.concatenate([np.asarray(objects[n]['x']) for n in names])
    y = np.concatenate([np.asarray(objects[n]['y']) for n in names])
    ends = np.cumsum([len(objects[n]['y']) for n in names])
    return X, y, {n: (e - len(objects[n]['y']), e) for n, e in zip(names, ends)}


def _loo_jobs(objects, **kw):
    """mr_gan.py:274-279: one job per held-out object."""
    X, y, spans = stack_objects(objects)
    rows = np.arange(len(y))
    jobs = []
    for name, (a, b) in spans.items():
        jobs.append(dict(X=X, y=y, train_idx=np.concatenate([rows[:a], rows[b:]]), test_idx=rows[a:b], name=name, **kw))
    return jobs


def job_rows(j):
    """(n_train, n_test) of a job in either format."""
    if 'train_idx' in j:
        return len(j['train_idx']), len(j['test_idx'])
    return len(j['trainTestSets'][0]), len(j['trainTestSets'][1])


def job_width(j):
    return j['X'].shape[1] if 'train_idx' in j else j['trainTestSets'][0].shape[1]


def job_cost(j):
    """Relative cost of a fold-training for the scheduler: the step is HBM-bound on the optimizer traffic, 28 bytes per
    parameter of N_D + N_G = 1501 D + 1 055 756 (SURVEY.md 8), i.e. ~ (D + 703) per step pair, times the pairs per epoch."""
    return (job_width(j) + 703.0) * max(job_rows(j)[0] // 50, 1)


def main(argv=None):
    parser = argparse.ArgumentParser(description='Semi-supervised learning with GANs for material recognition on haptic data.')
    parser.add_argument('-t', '--tables', nargs='+', help='[Required] Tables to recompute', required=True)
    parser.add_argument('-v', '--verbose', help='Verbose', action='store_true')
    # additive flags (defaults reproduce the reference's behaviour)
    parser.add_argument('--seed', type=int, default=None, help='seed for splits, initial weights, permutations and noise')
    parser.add_argument('--epochs', type=int, default=100)
    parser.add_argument('--precision', choices=['fp32', 'tf32', 'f16'], default='f16',
                        help='arithmetic of the dense layers: f16 = fp16 operand copies, fp32 accumulation and master weights (default; per-step '
                             'losses within 1e-3 of the oracle, 43 k step-pairs/s per B200); tf32; fp32 = FFMA parity mode (1e-7, 9.8 k)')
    parser.add_argument('--group', type=int, default=84,
                        help='largest number of folds trained side by side per handle (84 = two modalities of table 1; the GPU saturates at ~74 '
                             'folds of D=1200; results do not depend on it)')
    parser.add_argument('--data-dir', default='data_processed')
    parser.add_argument('--synthetic', action='store_true', help='synthetic data of the MREO shape instead of the processed pickles')
    parser.add_argument('--host-perm', action='store_true', help='draw the epoch permutations on the host (numpy) instead of on the device')
    results.add_arguments(parser, saliency=True)
    args = parser.parse_args(argv)
    rank, world, local = sweep.dist_env()
    seed = sweep.shared_seed(args.seed)          # one seed for every rank: same dataset, same splits, same job streams
    say = print if rank == 0 else (lambda *a, **k: None)
    if rank == 0:
        sys.stderr.write('seed: %d%s\n' % (seed, '   [SYNTHETIC data of the MREO shape: not the paper\'s dataset]' if args.synthetic else ''))
    jid = [0]
    rep = results.Report(args, 'mr_gan', rank, say, seed=seed, precision=args.precision, epochs=args.epochs)

    def run(jobs):
        for j in jobs:
            j['job_id'] = jid[0]
            jid[0] += 1
        res = sweep.run_sharded(
            jobs, lambda js, dev: train_gan_folds(js, epochs=args.epochs, verbose=args.verbose, seed=seed,
                                                  precision=args.precision, device=dev, device_perm=not args.host_perm,
                                                  details=rep.details, saliency=rep.saliency),
            group_size=args.group, key=job_rows, cost=job_cost)
        return res

    def report(errors, label='Average error:'):
        say(label, np.mean(errors), 'Average accuracy:', np.mean(1.0 - np.array(errors)))
        sys.stdout.flush()

    if '1' in args.tables:                      # mr_gan.py:244-261
        # every (modality, labeled %, fold) training is independent: all 294 are built first, sharded over the GPUs in one
        # go, and the results are printed afterwards in the reference's loop order
        percents = [1, 2, 4, 8, 16, 50, 100]
        jobs = []
        for modality in range(len(MODALITIES)):
            X, y = dataset(modalities=modality, seed=seed, data_dir=args.data_dir, synthetic_data=args.synthetic)
            jobs += [j for p in percents for j in _kfold_jobs(X, y, seed + p, percentlabeled=p)]
        res = run(jobs)
        errors = results.errors(res)
        say('\n', '-' * 25, 'Testing various amounts of labeled training data', '-' * 25)
        say('-' * 100)
        for modality in range(len(MODALITIES)):
            say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)
            for k, p in enumerate(percents):
                say('-' * 15, 'Percentage of training data labeled: %d%%' % p, '-' * 15)
                a = 42 * modality + 6 * k
                e = errors[a:a + 6]
                for v in e:
                    say('Test error:', v, 'Test accuracy:', 1.0 - v)
                report(e)
                rep.setting(jobs[a:a + 6], res[a:a + 6], synthetic.block_widths(modality), table=1, modality=MODALITIES[modality])

    if '3' in args.tables:                      # mr_gan.py:263-283
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
                report(errors[n * k:n * k + n], 'Average leave-one-object-out error:')
                rep.setting(jobs[n * k:n * k + n], res[n * k:n * k + n], synthetic.block_widths(modality), table=3,
                            modality=MODALITIES[modality])

    if '5' in args.tables:                      # mr_gan.py:285-318
        for header_mods, times, is_contact in (([0, 1, 2], [4, 3, 2, 1, 0.5, 0.2, 0.1], False),
                                               ([3], [1, 0.7, 0.5, 0.3, 0.2, 0.1, 0.05], True)):
            say('\n', '-' * 25, 'Testing various lengths of contact time in training data', '-' * 25)
            say('-' * 100)
            for modality in header_mods:
                say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)
                jobs = []
                for tm in times:
                    kw = dict(contactmicTime=tm) if is_contact else dict(forcetempTime=tm)
                    X, y = dataset(modalities=modality, seed=seed, data_dir=args.data_dir, synthetic_data=args.synthetic, **kw)
                    jobs += _kfold_jobs(X, y, seed, percentlabeled=100)
                res = run(jobs)
                errors = results.errors(res)
                for k, tm in enumerate(times):
                    say('-' * 15, 'Length of training data: %.1fs' % tm, '-' * 15)
                    for e in errors[6 * k:6 * k + 6]:
                        say('Test error:', e, 'Test accuracy:', 1.0 - e)
                    report(errors[6 * k:6 * k + 6])
                    kw = dict(contactmicTime=tm) if is_contact else dict(forcetempTime=tm)
                    rep.setting(jobs[6 * k:6 * k + 6], res[6 * k:6 * k + 6], synthetic.block_widths(modality, **kw), table=5,
                                modality=MODALITIES[modality], time=tm)

    if '6' in args.tables:                      # mr_gan.py:320-341
        say('\n', '-' * 25, 'Testing performance as quantity of unlabeled data increases', '-' * 25)
        say('-' * 100)
        for modality in [2, 5]:
            say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)
            X, y = dataset(modalities=modality, seed=seed, data_dir=args.data_dir, synthetic_data=args.synthetic)
            for percentlabeled in [4]:
                say('-' * 15, 'Percentage of training data labeled: %d%%' % percentlabeled, '-' * 15)
                unl = [0, 4, 8, 16, 32, 64, 100 - percentlabeled]
                jobs = [j for pu in unl for j in _kfold_jobs(X, y, seed + pu, percentlabeled=percentlabeled, percentunlabeled=pu)]
                res = run(jobs)
                errors = results.errors(res)
                for k, pu in enumerate(unl):
                    say('-' * 15, 'Percentage of training data unlabeled: %d%%' % pu, '-' * 15)
                    for e in errors[6 * k:6 * k + 6]:
                        say('Test error:', e, 'Test accuracy:', 1.0 - e)
                    report(errors[6 * k:6 * k + 6])
                    rep.setting(jobs[6 * k:6 * k + 6], res[6 * k:6 * k + 6], synthetic.block_widths(modality), table=6,
                                modality=MODALITIES[modality])
    rep.close()
    return 0


if __name__ == '__main__':
    sys.exit(main())
