"""Drop-in for the reference's ``mr_gan.py``: same ``dataset()`` / ``mr_gan()`` signatures,
same ``--tables`` CLI and stdout strings (mr_gan.py:236-341), with the compiled training step
(mr_gan.py:169-171) and the epoch loop (mr_gan.py:183-230) running as sm_100a CUDA behind the
C-ABI of include/mrgan.h.  New arguments are keyword-only and default to the reference's
behaviour.  No CPU fallback: without a B200 ``mr_gan()`` raises."""
import os
import sys
import time

import numpy as np

from . import checkpoint, foldprep, results, synthetic, tables
from .engine import FoldGroup
from .model import MATERIALS, init_disc, init_gen
from .tables import MODALITIES, job_rows, job_width, kfold_jobs, loo_jobs, stack_objects  # noqa: F401

_kfold_jobs, _loo_jobs = kfold_jobs, loo_jobs      # the names these had when they lived here (bench.py uses _kfold_jobs)


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
                    eval_each_epoch=True, shared_t=True, return_group=False, device_perm=False, details=False, saliency=False,
                    samples=False, start_states=None, on_epoch=None):
    """Train a GROUP of independent folds side by side on one GPU.

    jobs: list of dicts with keys ``trainTestSets`` (or ``X``, ``y``), ``percentlabeled``,
    ``percentunlabeled`` (optional), ``job_id`` (optional, seeds the fold's streams).
    device_perm: draw the epoch permutations of mr_gan.py:189-202 on the device (the host then sends one epoch number per
    epoch instead of 3 x int32[n_train] per fold); same distribution, different draws than the host's numpy generator.
    Returns the list of test errors (mr_gan.py:230,234), one per job; details=True: one dict per job instead,
    ``{'error': <the same float>, 'confusion': int32 [K, K]}`` (rows = true class, columns = predicted), from one extra
    forward pass over every fold's test set; saliency=True: those dicts with ``'saliency'``, float32 [K, D] (FoldGroup.saliency);
    samples=True: those dicts with ``'samples'`` (results.sample_report of FoldGroup.sample_stats) and ``'sample_rows'``, one
    batch of generated rows in raw feature units.  start_states / on_epoch: resume and snapshots (checkpoint.py)."""
    start = checkpoint.start_epoch(start_states, len(jobs))

    def init(fg, i, D, rng):
        if start_states is not None and start_states[i] is not None:
            return                                  # the weights come from the state
        fg.set_params(i, 1, init_gen(D, rng))       # generator first, as mr_gan.py:110-114 builds it first
        fg.set_params(i, 0, init_disc(D, rng))

    fg, folds, rngs = foldprep.load_folds(jobs, seed, lambda shapes: FoldGroup(
        shapes, model='gan', precision=precision, device=device, batch=batch, eval_each_epoch=eval_each_epoch,
        shared_t=shared_t), init, verbose)
    checkpoint.restore(fg, rngs, start_states)
    n_train = fg.shapes[0][1]
    if verbose:
        print('Epochs:', epochs)
        print('Batch size:', batch)
        print('Training batches per epoch:', n_train // batch)
        print('Testing batches per epoch:', fg.shapes[0][2] // batch)

    def draw():
        per = [foldprep.epoch_indices(rng, n_train, f.lab_rows, f.unl_rows) for f, rng in zip(folds, rngs)]
        return [np.stack([p[s] for p in per]) for s in range(3)]

    if device_perm and max(len(f.lab_rows) for f in folds) <= 8192 and all(
            (len(f.unl_rows) if f.unl_rows is not None else n_train) <= 8192 for f in folds):
        for i, f in enumerate(folds):
            fg.set_epoch_rows(i, f.lab_rows, f.unl_rows)
    else:
        device_perm = False
    nxt = None if device_perm or start >= epochs else draw()
    for epoch in range(start + 1, epochs + 1):
        begin = time.time()
        snap = None
        if device_perm:
            fg.train_epoch_seeded(epoch, wait=False)  # permutations drawn on the device from (fold key, epoch)
        else:
            fg.train_epoch(*nxt, wait=False)      # one CUDA-graph launch: the whole epoch, all folds
            if on_epoch is not None:
                snap = checkpoint.rng_states(rngs)  # the streams after this epoch's draws, before the next epoch's
            if epoch < epochs:
                nxt = draw()                      # host permutations of the next epoch overlap the GPU
        st = fg.epoch_result()
        if on_epoch is not None:
            on_epoch(epoch, fg, st, snap)
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
    errors = results.collect(fg, errors, details, saliency, samples=samples,
                             scalers=[checkpoint.job_scaler(j) for j in jobs] if samples else None)
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


def job_cost(j):
    """Relative cost of a fold-training for the scheduler: the step is HBM-bound on the optimizer traffic, 28 bytes per
    parameter of N_D + N_G = 1501 D + 1 055 756 (SURVEY.md 8), i.e. ~ (D + 703) per step pair, times the pairs per epoch."""
    return (job_width(j) + 703.0) * max(job_rows(j)[0] // 50, 1)


def main(argv=None):
    # --group 84 = two modalities of table 1; the GPU saturates at ~74 folds of D=1200
    parser = tables.argument_parser('Semi-supervised learning with GANs for material recognition on haptic data.', group=84)
    parser.add_argument('--host-perm', action='store_true', help='draw the epoch permutations on the host (numpy) instead of on the device')
    parser.add_argument('--samples', metavar='FILE', default=None,
                        help="write one batch of every fold-training's generated rows (raw feature units) to one .npz file (rank "
                             "0) and print the setting's sample statistics (Frechet distance and feature-matching gap of D's "
                             "layer-5 features, D's real-vs-fake score, predicted class shares) after its average")
    args = parser.parse_args(argv)

    def train(jobs, device, seed, rep, **resume):
        return train_gan_folds(jobs, epochs=args.epochs, verbose=args.verbose, seed=seed, precision=args.precision, device=device,
                               device_perm=not args.host_perm, details=rep.details, saliency=rep.saliency, samples=rep.samples,
                               **resume)

    return tables.run(args, 'mr_gan', train, job_rows, job_cost, ['1', '3', '5', '6'],
                      checkpoint_fields=dict(model='gan', shared_t=True, batch=50, perm='host' if args.host_perm else 'device'))


if __name__ == '__main__':
    sys.exit(main())
