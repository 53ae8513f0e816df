"""Saved GAN and NN fold-trainings: resume an interrupted training bitwise, and load a trained fold for inference.

One file per fold-training (``.npz``), so a file does not depend on how folds were grouped:

- ``meta``: one JSON string -- the fingerprint of the fold-training (``fingerprint``: format version, model, precision,
  ``shared_t``, batch, permutation mode, D, n_train, n_test, seed, job id, epochs asked for, labeled / unlabeled shares and
  a hash of the job's train / test rows), the config fields set beyond the defaults, the fold's Philox key, the epochs
  done and, with host permutations, the host stream's ``bit_generator.state`` after the last trained epoch's draws;
- ``p<net>``, ``m<net>``, ``v<net>``: the parameters and Adam's m and v of each net (0 = discriminator / classifier,
  1 = generator), flat in the reference's weight order; ``counters``: int32 [4] (include/mrgan.h, Checkpoints);
- ``x_test``, ``y_test``: the fold's resident scaled test set; ``scaler_mean``, ``scaler_scale``: float64, the fold's
  ``StandardScaler().fit(X[train_rows])``, so new raw rows can be classified (``LoadedModel.transform``).

Restoring the state into a fresh handle and training on gives bitwise what one uninterrupted run gives: noise comes from
Philox keyed by the fold key and the device step counter, device permutations are keyed by (fold key, epoch), and host
permutations come from the restored host stream."""
import copy
import hashlib
import json
import os
import tempfile

import numpy as np
from sklearn import preprocessing

from . import results
from .engine import PRECISION, FoldGroup
from .model import MATERIALS, NOISE_SIZE, disc_shapes, gen_shapes

FORMAT = 1
_PRECISION_NAME = {v: k for k, v in PRECISION.items()}


class CheckpointMismatch(ValueError):
    """A saved fold-training that is not the one this run would train (the message names the field)."""


def _job_rows(job):
    if 'train_idx' in job:
        return np.asarray(job['X']).shape[1], len(job['train_idx']), len(job['test_idx'])
    tts = job.get('trainTestSets')
    if tts is None:
        raise ValueError("a checkpoint needs a job with train_idx / test_idx or trainTestSets (the split must be known)")
    return np.shape(tts[0])[1], len(tts[0]), len(tts[1])


def rows_hash(job):
    """sha256 of what selects a job's rows: its train / test row indices, or the arrays of its trainTestSets."""
    h = hashlib.sha256()
    if 'train_idx' in job:
        parts = [np.asarray(job['train_idx'], np.int64), np.asarray(job['test_idx'], np.int64)]
    else:
        _job_rows(job)
        parts = [np.ascontiguousarray(a) for a in job['trainTestSets']]
    for a in parts:
        h.update(str((a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def fingerprint(job, *, model, precision, shared_t, batch, perm, seed, epochs):
    """The fields a saved fold-training must match to be resumed or reused (each is compared on its own)."""
    D, n_train, n_test = _job_rows(job)
    pu = job.get('percentunlabeled')
    return dict(format=FORMAT, model=model, precision=precision, shared_t=bool(shared_t), batch=int(batch), perm=perm,
                D=int(D), n_train=int(n_train), n_test=int(n_test), seed=int(seed), job_id=int(job.get('job_id', 0)),
                epochs=int(epochs), percentlabeled=job['percentlabeled'], percentunlabeled=pu, rows=rows_hash(job))


def check(meta, expected, path):
    """Raise CheckpointMismatch naming the first field of ``expected`` that ``meta`` does not match."""
    for k, want in expected.items():
        if meta.get(k) != want:
            raise CheckpointMismatch("checkpoint %s does not match this run: %s is %r in the file, %r here"
                                     % (path, k, meta.get(k), want))


def job_scaler(job):
    """The float64 StandardScaler (mean, scale) of a job's training rows (mr_gan.py:96-98)."""
    if 'train_idx' in job:
        x = np.asarray(job['X'])[np.asarray(job['train_idx'])]
    else:
        x = job['trainTestSets'][0]
    sc = preprocessing.StandardScaler().fit(np.asarray(x, dtype=np.float64))
    return np.asarray(sc.mean_, np.float64), np.asarray(sc.scale_, np.float64)


def save(path, fg, fold, job, *, seed, epochs, epochs_done, perm, rng_state=None):
    """Write fold ``fold`` of the group ``fg`` -- the training of ``job`` after ``epochs_done`` of ``epochs`` epochs -- to
    ``path`` (atomically: a reader sees the old file or the new one).  perm: 'device' or 'host' permutations; rng_state: the
    fold's host stream state after the last trained epoch's draws (host permutations)."""
    D, ntr, nte, key = fg.shapes[fold]
    meta = fingerprint(job, model=fg.model, precision=_PRECISION_NAME[fg.cfg.precision], shared_t=fg.cfg.shared_t,
                       batch=fg.batch, perm=perm, seed=seed, epochs=epochs)
    if (meta['D'], meta['n_train'], meta['n_test']) != (D, ntr, nte):
        raise ValueError("save: fold %d of the group is not the fold of this job" % fold)
    meta.update(config=dict(n_classes=int(fg.cfg.n_classes), eval_each_epoch=bool(fg.cfg.eval_each_epoch), **fg.hyper),
                key=int(key), epochs_done=int(epochs_done), rng_state=rng_state)
    st = fg.fold_state(fold)
    arrays = dict(counters=np.asarray(st['counters'], np.int32), x_test=fg.debug_buffer(fold, 51, nte, D))
    for i, net in enumerate(fg.nets):
        for k in ('params', 'm', 'v'):
            arrays['%s%d' % (k[0], net)] = np.concatenate([np.asarray(a, np.float32).ravel() for a in st[k][i]])
    y_test = np.asarray(job['y'])[np.asarray(job['test_idx'])] if 'train_idx' in job else job['trainTestSets'][3]
    arrays['y_test'] = np.asarray(y_test, np.int32)
    arrays['scaler_mean'], arrays['scaler_scale'] = job_scaler(job)
    d = os.path.dirname(os.path.abspath(path))
    fd, tmp = tempfile.mkstemp(prefix='.ckpt.', suffix='.tmp', dir=d)
    try:
        with os.fdopen(fd, 'wb') as f:
            np.savez(f, meta=np.array(json.dumps(meta)), **arrays)
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.unlink(tmp)
        raise


def read_meta(path):
    """The metadata of a saved fold-training; rejects a file of another format version."""
    with np.load(path, allow_pickle=False) as z:
        meta = json.loads(str(z['meta']))
    if meta.get('format') != FORMAT:
        raise CheckpointMismatch("checkpoint %s has format version %r; this version reads %d" % (path, meta.get('format'), FORMAT))
    return meta


def _net_shapes(meta, net):
    cfg = meta['config']
    if net == 0:
        return disc_shapes(meta['D'], cfg.get('n_classes', len(MATERIALS)))
    return gen_shapes(meta['D'], cfg.get('noise_dim', NOISE_SIZE))


def load_state(path):
    """A saved fold-training as a trainer's start state: ``FoldGroup.fold_state`` plus ``epochs_done``, ``rng_state`` and
    ``meta``."""
    meta = read_meta(path)
    nets = (0, 1) if meta['model'] == 'gan' else (0,)
    st = dict(params=[], m=[], v=[], epochs_done=meta['epochs_done'], rng_state=meta.get('rng_state'), meta=meta)
    with np.load(path, allow_pickle=False) as z:
        st['counters'] = np.asarray(z['counters'], np.int32)
        for net in nets:
            shp = _net_shapes(meta, net)
            for k in ('params', 'm', 'v'):
                flat = z['%s%d' % (k[0], net)]
                if flat.size != sum(int(np.prod(s)) for s in shp):
                    raise ValueError("checkpoint %s: %s of net %d has %d values, not the size of D=%d" % (path, k, net, flat.size, meta['D']))
                out, o = [], 0
                for s in shp:
                    n = int(np.prod(s))
                    out.append(flat[o:o + n].reshape(s).copy())
                    o += n
                st[k].append(out)
    return st


def start_epoch(states, n):
    """The epoch a group of n folds resumes after (0: none resumes); all folds of a group train in lockstep."""
    if states is None:
        return 0
    if len(states) != n:
        raise ValueError("start_states: one entry per job expected")
    done = {0 if s is None else int(s['epochs_done']) for s in states}
    if len(done) != 1:
        raise ValueError("start_states: the folds of one group must resume after the same epoch, not %s" % sorted(done))
    return done.pop()


def restore(fg, rngs, states):
    """Load each given state into its fold and set the fold's host stream to the saved state (host permutations)."""
    for i, st in enumerate(states or []):
        if st is None:
            continue
        fg.load_fold_state(i, st)
        if st.get('rng_state') is not None:
            rngs[i].bit_generator.state = st['rng_state']


def rng_states(rngs):
    return [copy.deepcopy(r.bit_generator.state) for r in rngs]


class LoadedModel(FoldGroup):
    """A one-fold inference group of a saved fold-training: ``predict``, ``predict_rows``, ``confusion``, ``eval``,
    ``test_error``, ``input_grad``, ``saliency``, ``generate`` and ``sample_stats`` work as on the live group; ``transform``
    scales raw rows and ``inverse_transform`` returns scaled rows (a generated sample) to raw feature units."""

    def transform(self, X_raw):
        """Raw feature rows [n, D] -> the fold's scaled input space (the saved scaler, float64, then float32)."""
        x = np.asarray(X_raw, dtype=np.float64)
        if x.ndim != 2 or x.shape[1] != self.scaler_mean.size:
            raise ValueError("transform: X_raw must be [n, %d]" % self.scaler_mean.size)
        return ((x - self.scaler_mean) / self.scaler_scale).astype(np.float32)

    def inverse_transform(self, x):
        """Scaled rows [n, D] (e.g. generate()'s) -> raw feature units, float64 (the saved scaler)."""
        x = np.asarray(x, dtype=np.float64)
        if x.ndim != 2 or x.shape[1] != self.scaler_mean.size:
            raise ValueError("inverse_transform: x must be [n, %d]" % self.scaler_mean.size)
        return x * self.scaler_scale + self.scaler_mean


def load_model(path, device=0):
    """The saved fold-training at ``path`` as a LoadedModel on ``device``: a handle of the saved shape holding the saved
    test set, a zero training block of one batch and the saved weights.  No training data is needed."""
    st = load_state(path)
    meta = st['meta']
    cfg = dict(meta['config'])
    D, nte, B = meta['D'], meta['n_test'], meta['batch']
    fg = LoadedModel([(D, B, nte, meta['key'])], model=meta['model'], precision=meta['precision'], device=device, batch=B,
                     shared_t=meta['shared_t'], n_classes=cfg.pop('n_classes'), eval_each_epoch=cfg.pop('eval_each_epoch'),
                     **cfg)
    try:
        with np.load(path, allow_pickle=False) as z:
            fg.scaler_mean, fg.scaler_scale = z['scaler_mean'], z['scaler_scale']
            fg.load_fold(0, np.zeros((B, D), np.float32), np.zeros(B, np.int32), z['x_test'], z['y_test'])
        fg.load_fold_state(0, st)
        fg.meta = meta
        return fg
    except BaseException:
        fg.close()
        raise


class Sweep:
    """``--checkpoint DIR`` of a table CLI: per job ``DIR/<tool>_job<id>.npz``.  ``start(job)`` reads and checks a job's
    file (metadata only) and returns the epochs it has done (0 without a file); ``train`` trains a group of jobs that resume
    after the same epoch, writing their state every ``every`` epochs and at the end, or, for files that are final, takes
    the results from the loaded models."""

    def __init__(self, directory, tool, seed, epochs, every, fields):
        self.dir, self.tool, self.seed, self.epochs, self.every, self.fields = directory, tool, seed, epochs, every or 0, fields
        os.makedirs(directory, exist_ok=True)
        self.done = {}

    def path(self, job):
        return os.path.join(self.dir, '%s_job%d.npz' % (self.tool, job['job_id']))

    def expected(self, job):
        return fingerprint(job, seed=self.seed, epochs=self.epochs, **self.fields)

    def start(self, job):
        p = self.path(job)
        done = 0
        if os.path.exists(p):
            meta = read_meta(p)
            check(meta, self.expected(job), p)
            done = int(meta['epochs_done'])
        self.done[job['job_id']] = done
        return done

    def train(self, jobs, device, rep, train):
        """train(jobs, device, seed, rep, start_states=..., on_epoch=...): the CLI's trainer."""
        done = self.done[jobs[0]['job_id']]
        if done >= self.epochs:
            out = []
            for j in jobs:
                with load_model(self.path(j), device) as fg:
                    out += results.collect(fg, [fg.test_error(0)], rep.details, rep.saliency, samples=getattr(rep, 'samples', False),
                                           scalers=[(fg.scaler_mean, fg.scaler_scale)])
            return out
        states = [load_state(self.path(j)) for j in jobs] if done else None

        def on_epoch(epoch, fg, stats, rngs):
            if epoch == self.epochs or (self.every and epoch % self.every == 0):
                for i, j in enumerate(jobs):
                    save(self.path(j), fg, i, j, seed=self.seed, epochs=self.epochs, epochs_done=epoch,
                         perm=self.fields['perm'], rng_state=None if rngs is None else rngs[i])
        return train(jobs, device, self.seed, rep, start_states=states, on_epoch=on_epoch)

