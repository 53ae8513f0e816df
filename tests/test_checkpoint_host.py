"""CPU suite of checkpoints (mr_gan_b200/checkpoint.py) with a fake fold group: the file format round trip and the rejection
of another format version, the fingerprint error for each field, the table CLIs without --checkpoint, the start epoch in
the grouping key, and the new C-ABI symbols in both the header and the binding."""
import json
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

from mr_gan_b200 import _lib, checkpoint, mr_gan, mr_nn
from mr_gan_b200.model import disc_shapes, gen_shapes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D, NTR, NTE = 8, 60, 12


def _job(job_id=3, **kw):
    rng = np.random.default_rng(job_id)
    X = rng.standard_normal((NTR + NTE, D)).astype(np.float32)
    y = np.arange(NTR + NTE) % 6
    return dict(X=X, y=y, train_idx=np.arange(NTR), test_idx=np.arange(NTR, NTR + NTE), percentlabeled=4, job_id=job_id, **kw)


class FakeGroup:
    """What checkpoint.save reads of a FoldGroup, for one GAN fold of width D."""
    model, nets, batch, hyper = 'gan', (0, 1), 50, {'sigma_in': 0.25}
    cfg = SimpleNamespace(precision=2, shared_t=1, n_classes=6, eval_each_epoch=1)

    def __init__(self):
        self.shapes = [(D, NTR, NTE, 12345)]
        rng = np.random.default_rng(0)
        self.state = dict(counters=np.array([24, 0, 0, 48], np.int32), params=[], m=[], v=[])
        for shp in (disc_shapes(D), gen_shapes(D)):
            for k in ('params', 'm', 'v'):
                self.state[k].append([rng.standard_normal(s).astype(np.float32) for s in shp])
        self.x_test = rng.standard_normal((NTE, D)).astype(np.float32)

    def fold_state(self, fold):
        return self.state

    def debug_buffer(self, fold, which, rows, cols):
        assert (which, rows, cols) == (51, NTE, D)
        return self.x_test


def test_format_round_trip_and_unknown_version(tmp_path):
    fg, job = FakeGroup(), _job()
    rng = np.random.default_rng([1, 2])
    rng.permutation(10)
    path = str(tmp_path / 'f.npz')
    checkpoint.save(path, fg, 0, job, seed=1, epochs=6, epochs_done=2, perm='host', rng_state=rng.bit_generator.state)
    meta = checkpoint.read_meta(path)
    checkpoint.check(meta, checkpoint.fingerprint(job, model='gan', precision='f16', shared_t=True, batch=50, perm='host',
                                                  seed=1, epochs=6), path)
    assert meta['epochs_done'] == 2 and meta['key'] == 12345 and meta['config'] == dict(n_classes=6, eval_each_epoch=True, sigma_in=0.25)
    st = checkpoint.load_state(path)
    assert np.array_equal(st['counters'], fg.state['counters'])
    for k in ('params', 'm', 'v'):
        for a, b in zip(st[k], fg.state[k]):
            assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    r2 = np.random.default_rng(0)
    r2.bit_generator.state = st['rng_state']
    assert np.array_equal(r2.permutation(50), rng.permutation(50))           # the host stream continues where it stopped
    with np.load(path) as z:
        assert np.array_equal(z['x_test'], fg.x_test) and np.array_equal(z['y_test'], job['y'][job['test_idx']])
        mean, scale = z['scaler_mean'], z['scaler_scale']
    from sklearn.preprocessing import StandardScaler
    sc = StandardScaler().fit(job['X'][job['train_idx']].astype(np.float64))
    assert mean.dtype == np.float64 and np.array_equal(mean, sc.mean_) and np.array_equal(scale, sc.scale_)
    # another format version is refused by every reader
    with np.load(path) as z:
        arrays = {k: z[k] for k in z.files}
    meta['format'] = checkpoint.FORMAT + 1
    arrays['meta'] = np.array(json.dumps(meta))
    np.savez(path, **arrays)
    for read in (checkpoint.read_meta, checkpoint.load_state):
        with pytest.raises(checkpoint.CheckpointMismatch, match='format version'):
            read(path)


FIELDS = dict(model='gan', precision='f16', shared_t=True, batch=50, perm='device', seed=0, epochs=4)


@pytest.mark.parametrize("field,other", [
    ('model', dict(model='nn')), ('precision', dict(precision='fp32')), ('shared_t', dict(shared_t=False)),
    ('batch', dict(batch=20)), ('perm', dict(perm='host')), ('seed', dict(seed=1)), ('epochs', dict(epochs=5)),
    ('job_id', dict(job_id=4)), ('percentlabeled', dict(percentlabeled=8)), ('percentunlabeled', dict(percentunlabeled=16)),
    ('D', dict(D=9)), ('n_test', dict(n_test=11)), ('rows', dict(rows=True))])
def test_fingerprint_mismatch_names_the_field(field, other):
    job = _job()
    meta = checkpoint.fingerprint(job, **FIELDS)
    kw = {k: v for k, v in other.items() if k in FIELDS}
    j2 = dict(job)
    if field in ('job_id', 'percentlabeled', 'percentunlabeled'):
        j2[field] = other[field]
    elif field == 'D':
        j2['X'] = np.zeros((NTR + NTE, 9), np.float32)
    elif field == 'n_test':
        j2['test_idx'] = job['test_idx'][:11]
    elif field == 'rows':
        j2['train_idx'] = job['train_idx'][::-1]
    want = checkpoint.fingerprint(j2, **dict(FIELDS, **kw))
    with pytest.raises(checkpoint.CheckpointMismatch, match=r'does not match this run: %s is ' % field):
        checkpoint.check(meta, want, 'f.npz')
    checkpoint.check(meta, checkpoint.fingerprint(job, **FIELDS), 'f.npz')


@pytest.mark.parametrize("mod,fn,table", [(mr_gan, 'train_gan_folds', '6'), (mr_nn, 'train_nn_folds', '2')])
def test_without_checkpoint_the_trainers_get_todays_call(mod, fn, table, monkeypatch, capsys):
    seen = []

    def spy(js, *a, **kw):
        seen.append(set(kw))
        return [0.25] * len(js)

    monkeypatch.setattr(mod, fn, spy)
    assert mod.main(['--tables', table, '--synthetic', '--seed', '0']) == 0
    assert seen and not any({'start_states', 'on_epoch'} & k for k in seen)
    assert 'Average error: 0.25' in capsys.readouterr().out


def test_start_epoch_enters_the_grouping_key(monkeypatch, tmp_path, capsys):
    """Jobs that resume after different epochs never share a group; the rest still group by the CLI's own key."""
    starts = {}
    groups = []

    def start(self, job):
        self.done[job['job_id']] = starts[job['job_id']] = (job['job_id'] % 3) * 2     # 0, 2 or 4 (= final)
        return starts[job['job_id']]

    def train(self, jobs, device, rep, trainer):
        groups.append([j['job_id'] for j in jobs])
        return [0.5] * len(jobs)

    monkeypatch.setattr(checkpoint.Sweep, 'start', start)
    monkeypatch.setattr(checkpoint.Sweep, 'train', train)
    assert mr_nn.main(['--tables', '2', '--synthetic', '--seed', '0', '--epochs', '4', '--checkpoint', str(tmp_path)]) == 0
    assert sorted(i for g in groups for i in g) == sorted(starts)
    assert all(len({starts[i] for i in g}) == 1 for g in groups)
    assert {starts[g[0]] for g in groups} == {0, 2, 4}
    assert 'Average error: 0.5' in capsys.readouterr().out


def test_checkpoint_every_needs_checkpoint():
    with pytest.raises(SystemExit, match='needs --checkpoint'):
        mr_nn.main(['--tables', '2', '--synthetic', '--seed', '0', '--checkpoint-every', '2'])


def test_new_symbols_in_header_and_binding():
    with open(os.path.join(ROOT, 'include', 'mrgan.h')) as f:
        header = f.read()
    for name in ('mrgan_set_adam', 'mrgan_get_fold_counters', 'mrgan_set_fold_counters'):
        assert re.search(r'\b%s\(' % name, header), name
        assert name in _lib.SYMBOLS
    assert _lib.ABI_VERSION == 3 and '#define MRGAN_ABI_VERSION 3' in header
