"""GPU tier of checkpoints (mr_gan_b200/checkpoint.py): a GAN / NN training saved after 3 of 6 epochs and restored into fresh
handles, in another fold order and grouping, ends bitwise where the uninterrupted run ends; a model loaded in a new process
predicts bitwise like the live group; the new entry points reject bad calls; and the table CLIs resumed from a mix of final,
intermediate and missing files print what an uninterrupted run prints."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from mr_gan_b200 import _lib, checkpoint, mr_gan, mr_nn
from mr_gan_b200.engine import FoldGroup, MrganError

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARG, STATE = -1, -4
WIDTHS = (400, 1200, 2432)
N, NTR = 720, 600                      # 120 test rows; 600 training rows = 12 GAN batches / 30 NN batches


def _jobs(percentlabeled=4):
    """Three index jobs of different width and equal n_train, balanced classes."""
    out = []
    for k, D in enumerate(WIDTHS):
        rng = np.random.default_rng(100 + k)
        y = np.arange(N) % 6
        X = (rng.standard_normal((N, D)) + y[:, None] * 0.05).astype(np.float32)
        perm = rng.permutation(N)
        out.append(dict(X=X, y=y, train_idx=np.sort(perm[:NTR]), test_idx=np.sort(perm[NTR:]), percentlabeled=percentlabeled,
                        job_id=10 + k))
    return out


def _run(train, jobs, epochs, start_states=None, save_to=None, perm=None, **kw):
    """Train; returns the per-epoch stats by epoch and, at the last epoch, the fold states, errors, confusion and saliency,
    folds in the order of jobs.  save_to: one path per job, written at the last epoch (checkpoint.save, 6 epochs asked for)."""
    rec = {'stats': {}}

    def on_epoch(epoch, fg, st, rngs):
        rec['stats'][epoch] = st.copy()
        if epoch == epochs:
            rec['states'] = [fg.fold_state(i) for i in range(len(jobs))]
            rec['err'] = [fg.test_error(i) for i in range(len(jobs))]
            rec['conf'] = fg.confusion()
            rec['sal'] = fg.saliency()
            for i, p in enumerate(save_to or []):
                checkpoint.save(p, fg, i, jobs[i], seed=7, epochs=6, epochs_done=epoch, perm=perm,
                                rng_state=None if rngs is None else rngs[i])
    train(jobs, epochs=epochs, seed=7, start_states=start_states, on_epoch=on_epoch, **kw)
    return rec


def _same_state(a, b):
    assert np.array_equal(a['counters'], b['counters']), (a['counters'], b['counters'])
    for k in ('params', 'm', 'v'):
        for na, nb in zip(a[k], b[k]):
            for x, y in zip(na, nb):
                assert x.tobytes() == y.tobytes(), k


def _resume_check(train, tmp_path, perm, **kw):
    """6 epochs straight against 3 epochs, saved, and 3 more in new handles: fold 2 alone, then folds 1 and 0 together."""
    jobs = _jobs()
    straight = _run(train, jobs, 6, **kw)
    paths = [str(tmp_path / ('job%d.npz' % i)) for i in range(len(jobs))]
    _run(train, jobs, 3, save_to=paths, perm=perm, **kw)
    got = {}
    for grp in ([2], [1, 0]):
        r = _run(train, [jobs[g] for g in grp], 6, start_states=[checkpoint.load_state(paths[g]) for g in grp], **kw)
        for n, g in enumerate(grp):
            got[g] = dict(state=r['states'][n], err=r['err'][n], conf=r['conf'][n], sal=r['sal'][n],
                          stats={e: r['stats'][e][n] for e in (4, 5, 6)})
        assert sorted(r['stats']) == [4, 5, 6]
    for g in range(3):
        _same_state(got[g]['state'], straight['states'][g])
        for e in (4, 5, 6):
            assert got[g]['stats'][e].tobytes() == straight['stats'][e][g].tobytes(), (g, e)
        assert got[g]['err'] == straight['err'][g]
        assert np.array_equal(got[g]['conf'], straight['conf'][g])
        assert got[g]['sal'].tobytes() == straight['sal'][g].tobytes()


@pytest.mark.parametrize("precision", ["fp32", "tf32", "f16"])
def test_gan_resume_bitwise_device_perm(precision, tmp_path):
    _resume_check(mr_gan.train_gan_folds, tmp_path, 'device', precision=precision, device_perm=True)


def test_gan_resume_bitwise_host_perm(tmp_path):
    _resume_check(mr_gan.train_gan_folds, tmp_path, 'host', precision='f16', device_perm=False)


def test_gan_resume_bitwise_separate_counters(tmp_path):
    _resume_check(mr_gan.train_gan_folds, tmp_path, 'device', precision='f16', device_perm=True, shared_t=False)


@pytest.mark.parametrize("precision", ["fp32", "tf32", "f16"])
def test_nn_resume_bitwise(precision, tmp_path):
    _resume_check(mr_nn.train_nn_folds, tmp_path, 'host', precision=precision, batch=20)


LOADER = r"""
import sys
sys.path.insert(0, %r)
import numpy as np
from mr_gan_b200 import checkpoint
d = np.load(%r)
with checkpoint.load_model(%r) as fg:
    pred, logits = fg.predict(0)
    rows_pred, rows_logits = fg.predict_rows(0, fg.transform(d['x_raw']))
    np.savez(%r, pred=pred, logits=logits, conf=fg.confusion(), err=np.float64(fg.test_error(0)), ev=np.float32(fg.eval(0)),
             sal=fg.saliency()[0], grad=fg.input_grad(0, d['x_few']), rows_pred=rows_pred, rows_logits=rows_logits)
print("OK")
"""


@pytest.mark.parametrize("model", ["gan", "nn"])
def test_loaded_model_equals_live_model(model, tmp_path):
    job = _jobs()[1]
    path = str(tmp_path / 'model.npz')
    live = {}

    def on_epoch(epoch, fg, st, rngs):
        if epoch == 2:
            checkpoint.save(path, fg, 0, job, seed=3, epochs=2, epochs_done=2, perm='host', rng_state=rngs[0])
            live['pred'], live['logits'] = fg.predict(0)
            live.update(conf=fg.confusion(), err=fg.test_error(0), ev=fg.eval(0), sal=fg.saliency()[0])
            live['x_few'] = fg.debug_buffer(0, 51, 5, job['X'].shape[1])
            live['grad'] = fg.input_grad(0, live['x_few'])

    train = mr_gan.train_gan_folds if model == 'gan' else mr_nn.train_nn_folds
    train([job], epochs=2, seed=3, precision='f16', on_epoch=on_epoch)
    inp, out = str(tmp_path / 'in.npz'), str(tmp_path / 'out.npz')
    np.savez(inp, x_raw=job['X'][job['test_idx']], x_few=live['x_few'])
    r = subprocess.run([sys.executable, '-c', LOADER % (ROOT, inp, path, out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'OK' in r.stdout, r.stdout + r.stderr
    got = np.load(out)
    for k in ('pred', 'logits', 'conf', 'sal', 'grad'):
        assert got[k].tobytes() == np.asarray(live[k]).tobytes(), k
    assert float(got['err']) == live['err'] and got['ev'] == live['ev']
    # new raw rows through the saved scaler: float64 scaling may round a last bit differently from the device's
    np.testing.assert_allclose(got['rows_logits'], live['logits'], rtol=1e-5, atol=1e-5)
    top2 = np.sort(live['logits'], axis=1)[:, -2:]
    differ = got['rows_pred'] != live['pred']
    assert np.all(top2[differ, 1] - top2[differ, 0] < 1e-5 * np.maximum(1.0, np.abs(top2[differ, 1])))


def test_entry_points_reject_bad_calls():
    """In the style of test_gpu_entry_guard.py: status and a key phrase of mrgan_last_error; the handle stays usable."""
    lib = _lib.load()
    D, NT, NE = 16, 100, 20
    x = np.zeros((NT, D), np.float32)
    y = (np.arange(NT) % 6).astype(np.int32)
    g = FoldGroup([(D, NT, NE, 1)])
    s = FoldGroup([(D, NT, NE, 1)], model='svm')
    v = FoldGroup([(D, NT, NE, 5)] * 2, batch=20)
    v.dp_init_virtual(2)
    try:
        n = g.num_params(0, 0)
        buf, cnt, neg = np.zeros(n + 8, np.float32), np.zeros(4, np.int32), np.array([0, 0, -1, 0], np.int32)
        fp, ip = _lib.fptr(buf), _lib.iptr(cnt)
        nets, dp = 'not available on an SVM handle', 'not available on a data-parallel handle'
        cases = [
            (g, lambda h: lib.mrgan_set_adam(h, 0, 0, fp, fp, n - 1), ARG, 'length does not match'),
            (g, lambda h: lib.mrgan_set_adam(h, 0, 0, fp, None, n), ARG, 'null pointer'),
            (g, lambda h: lib.mrgan_set_adam(h, 0, 2, fp, fp, n), ARG, 'no such net'),
            (g, lambda h: lib.mrgan_set_adam(h, 1, 0, fp, fp, n), ARG, 'fold index out of range'),
            (g, lambda h: lib.mrgan_get_fold_counters(h, 0, None), ARG, 'null pointer'),
            (g, lambda h: lib.mrgan_set_fold_counters(h, 0, None), ARG, 'null pointer'),
            (g, lambda h: lib.mrgan_set_fold_counters(h, 0, _lib.iptr(neg)), ARG, 'negative counter'),
            (None, lambda h: lib.mrgan_set_fold_counters(h, 0, ip), ARG, 'null handle'),
            (None, lambda h: lib.mrgan_get_fold_counters(h, 0, ip), ARG, 'null handle'),
            (None, lambda h: lib.mrgan_set_adam(h, 0, 0, fp, fp, n), ARG, 'null handle'),
            (s, lambda h: lib.mrgan_set_adam(h, 0, 0, fp, fp, n), STATE, nets),
            (s, lambda h: lib.mrgan_get_fold_counters(h, 0, ip), STATE, nets),
            (s, lambda h: lib.mrgan_set_fold_counters(h, 0, ip), STATE, nets),
            (v, lambda h: lib.mrgan_set_adam(h, 0, 0, fp, fp, n), STATE, dp),
            (v, lambda h: lib.mrgan_get_fold_counters(h, 0, ip), STATE, dp),
            (v, lambda h: lib.mrgan_set_fold_counters(h, 0, ip), STATE, dp),
        ]
        for k, (fg, call, code, phrase) in enumerate(cases):
            h = fg._h if fg is not None else None
            got = call(h)
            msg = lib.mrgan_last_error(h).decode()
            assert got == code and phrase in msg, (k, got, msg)
        # the handle stays usable: counters and a state round trip, then an evaluation
        g.load_fold(0, x, y, x[:NE], y[:NE])
        g.set_fold_counters(0, [7, 3, 4, 9])
        assert list(g.fold_counters(0)) == [7, 3, 4, 9] and g.counters(0) == (7, 9)
        st = g.fold_state(0)
        g.load_fold_state(0, st)
        _same_state(g.fold_state(0), st)
        g.eval(0)
        with pytest.raises(ValueError):
            g.load_fold_state(0, dict(st, counters=np.zeros(3, np.int32)))
        with pytest.raises(MrganError):
            g.set_fold_counters(0, [0, -1, 0, 0])
    finally:
        for fg in (g, s, v):
            fg.close()


def test_restore_between_epochs_needs_no_recapture():
    """The epoch graph reads the counters from device memory: after a restore the next epochs launch exactly the kernels
    of an epoch before it (a recapture would add the capture's launches)."""
    seen = []

    def on_epoch(epoch, fg, st, rngs):
        seen.append(fg.kernel_launches)
        if epoch == 2:
            fg.load_fold_state(0, fg.fold_state(0))
            seen.append(fg.kernel_launches)

    mr_gan.train_gan_folds(_jobs()[:1], epochs=4, seed=1, precision='f16', device_perm=True, on_epoch=on_epoch)
    e1, e2, r, e3, e4 = seen
    assert e3 - r == e2 - e1 == e4 - e3, seen


def _cli(mod, argv, cwd):
    r = subprocess.run([sys.executable, '-c', 'import sys; sys.path.insert(0, %r); from mr_gan_b200 import %s as m; '
                        'sys.exit(m.main(sys.argv[1:]))' % (ROOT, mod)] + argv, capture_output=True, text=True, cwd=cwd,
                       timeout=3000)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


KEEP_EPOCH2 = r"""
import os, shutil, sys
sys.path.insert(0, %r)
from mr_gan_b200 import checkpoint, %s as m
save = checkpoint.save
def keep(path, *a, **kw):
    save(path, *a, **kw)
    if kw['epochs_done'] == 2 and os.path.basename(path) in %r:
        shutil.copy(path, path + '.epoch2')
checkpoint.save = keep
sys.exit(m.main(sys.argv[1:]))
"""


@pytest.mark.parametrize("mod,table", [("mr_gan", "6"), ("mr_nn", "2")])
def test_cli_resume_prints_what_an_uninterrupted_run_prints(mod, table, tmp_path):
    d = tmp_path / 'ck'
    base = ['--tables', table, '--synthetic', '--seed', '0', '--epochs', '4', '--confusion']
    resumed_jobs, missing_jobs = [3, 40, 77], [5, 41]
    names = ['%s_job%d.npz' % (mod, i) for i in resumed_jobs]
    r = subprocess.run([sys.executable, '-c', KEEP_EPOCH2 % (ROOT, mod, names)] + base +
                       ['--checkpoint', str(d), '--checkpoint-every', '2'], capture_output=True, text=True, timeout=3000)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    first = r.stdout
    for n in names:                                         # only the epoch-2 state remains
        shutil.move(str(d / (n + '.epoch2')), str(d / n))
        assert checkpoint.read_meta(str(d / n))['epochs_done'] == 2
    for i in missing_jobs:
        os.unlink(str(d / ('%s_job%d.npz' % (mod, i))))
    rerun = _cli(mod, base + ['--checkpoint', str(d)], str(tmp_path))
    plain = _cli(mod, base, str(tmp_path))
    assert rerun == first
    assert plain == first
    for i in resumed_jobs + missing_jobs:
        assert checkpoint.read_meta(str(d / ('%s_job%d.npz' % (mod, i))))['epochs_done'] == 4
    # a file of another run is an error that names the field, and is left as it is
    p = d / ('%s_job0.npz' % mod)
    before = p.read_bytes()
    other = ['--tables', table, '--synthetic', '--seed', '0', '--epochs', '5', '--checkpoint', str(d)]
    r = subprocess.run([sys.executable, '-c', 'import sys; sys.path.insert(0, %r); from mr_gan_b200 import %s as m; '
                        'sys.exit(m.main(sys.argv[1:]))' % (ROOT, mod)] + other, capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and 'epochs is 4 in the file, 5 here' in r.stderr, r.stderr[-2000:]
    assert p.read_bytes() == before
