"""Drop-in for the reference's ``mr_nn.py``: the fully-supervised dense classifier (same
discriminator architecture, MSE vs one-hot, default Adam, batch 20; mr_nn.py:69-119) and its
``--tables 2 4`` CLI (mr_nn.py:121-168), on the same sm_100a kernels as the GAN path."""
import sys

import numpy as np

from . import foldprep, results, tables
from .engine import FoldGroup
from .model import init_disc
from .tables import job_rows, job_width


def train_nn_folds(jobs, epochs=100, verbose=False, *, seed=0, precision='f16', device=0, batch=20, details=False, saliency=False):
    """Train a group of independent mr_nn folds side by side; returns test errors (mr_nn.py:118-119), or with details=True
    one dict per job, ``{'error': <the same float>, 'confusion': int32 [K, K]}`` (rows = true class, columns = predicted);
    saliency=True: those dicts with ``'saliency'``, float32 [K, D] (FoldGroup.saliency)."""
    fg, folds, rngs = foldprep.load_folds(
        jobs, seed, lambda shapes: FoldGroup(shapes, model='nn', precision=precision, device=device, batch=batch),
        lambda fg, i, D, rng: fg.set_params(i, 0, init_disc(D, rng)), verbose, same_labeled=True)
    try:
        n_lab = len(folds[0].lab_rows)
        if n_lab % batch:
            raise ValueError("labeled rows (%d) must be a multiple of the batch size (%d)" % (n_lab, batch))

        def draw():   # model.fit(shuffle=True): one permutation of the labeled rows per epoch (mr_nn.py:117)
            return np.stack([f.lab_rows[rng.permutation(n_lab)] for f, rng in zip(folds, rngs)]).astype(np.int32)

        nxt = draw()
        for epoch in range(epochs):
            fg.nn_train_epoch(nxt, wait=False)
            if epoch + 1 < epochs:
                nxt = draw()
        errors = [1.0 - float(fg.nn_evaluate(i)[1]) for i in range(len(jobs))]     # mr_nn.py:118
        return results.collect(fg, errors, details, saliency)
    finally:
        fg.close()


def mr_nn(X, y, percentlabeled=50, trainTestSets=None, verbose=False, *, seed=None, epochs=100, precision='f16',
          device=0):
    """mr_nn.py:69-119, one fold."""
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))      # mr_nn.py:70-71
    job = dict(X=X, y=y, percentlabeled=percentlabeled, trainTestSets=trainTestSets)
    return train_nn_folds([job], epochs=epochs, verbose=verbose, seed=seed, precision=precision, device=device)[0]


def main(argv=None):
    args = tables.argument_parser('Collecting data from a spinning platter of objects.', group=42).parse_args(argv)

    def train(jobs, device, seed, rep):
        return train_nn_folds(jobs, epochs=args.epochs, verbose=args.verbose, seed=seed, precision=args.precision, device=device,
                              details=rep.details, saliency=rep.saliency)

    return tables.run(args, 'mr_nn', train, lambda j: job_rows(j) + (j['percentlabeled'],),
                      lambda j: job_width(j) * j['percentlabeled'], ['2', '4'])


if __name__ == '__main__':
    sys.exit(main())
