"""GPU tier of the generator samples (mrgan_generate, mrgan_sample_stats): parity with the oracle's generator on the weights
read back, the device z stream, independence of the batch chunking and the fold grouping, the statistics against
predict_rows and numpy, bitwise reproducibility, no side effects on later results, error codes, loaded checkpoints and the
mr_gan CLI's --samples."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from mr_gan_b200 import _lib, checkpoint, mr_gan
from mr_gan_b200.engine import TID_GEN, FoldGroup
from oracle import gan_oracle as O
from oracle import philox

from test_gpu_predict import NTE, NTR, K, _folds, _group

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 50                     # the fixtures' GAN batch; NE = max(3 B, n_test) = 150 rows per chunk


def _key(seed):
    return (seed & 0xFFFFFFFF, seed >> 32)


def _sig_lse(logits):
    l = np.asarray(logits, np.float64)
    m = l.max(axis=1)
    lse = m + np.log(np.exp(l - m[:, None]).sum(axis=1))
    return 1.0 / (1.0 + np.exp(-lse))


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 7e-4), ("f16", 7e-4)])
def test_generate_matches_oracle(precision, tol):
    """Rows of 300 = 2 chunks against gan_oracle.gen_forward per 50-row batch, on the weights read back and z replayed by
    oracle.philox: fp32 max error relative to the batch's largest |x|; tf32 / f16 norm-wise."""
    folds = _folds((400, 1200))
    n, seed = 6 * B, 11
    with _group('gan', precision, folds) as fg:
        worst = 0.0
        for i, f in enumerate(folds):
            x = fg.generate(i, n, seed=seed)
            assert x.shape == (n, f['D']) and x.dtype == np.float32
            pG = [np.asarray(a, np.float64) for a in fg.get_params(i, 1)]
            z = philox.normal(_key(f['seed']), seed, TID_GEN, n, fg.noise_dim)
            for b in range(0, n, B):
                ref, _ = O.gen_forward(pG, z[b:b + B])
                got = x[b:b + B].astype(np.float64)
                err = (np.abs(got - ref).max() / np.abs(ref).max() if precision == 'fp32'
                       else np.linalg.norm(got - ref) / np.linalg.norm(ref))
                worst = max(worst, err)
        print("MEASURED generate %s %.3g" % (precision, worst))
        assert worst <= tol


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_z_stream_and_chunk_independence(precision):
    """generate(seed=s) = generate(z = fill_normal(fold, s, TID_GEN, n, noise_dim)); rows [kB, (k+1)B) of a 6B request (two
    chunks) = generate(z = that slice): BatchNorm statistics per batch, nothing depends on the chunk."""
    folds = _folds((400, 1200))
    n, seed = 6 * B, 5
    with _group('gan', precision, folds) as fg:
        for i in range(2):
            x = fg.generate(i, n, seed=seed)
            z = fg.fill_normal(i, seed, TID_GEN, n, fg.noise_dim)
            assert fg.generate(i, n, z=z).tobytes() == x.tobytes()
            for k in range(n // B):
                assert fg.generate(i, B, z=z[k * B:(k + 1) * B]).tobytes() == x[k * B:(k + 1) * B].tobytes(), (i, k)
            assert fg.generate(i, n, seed=seed + 1).tobytes() != x.tobytes()


@pytest.mark.parametrize("precision", ["fp32", "tf32", "f16"])
def test_stats_against_predict_rows_and_numpy(precision):
    folds = _folds((400, 1200))
    with _group('gan', precision, folds) as fg:
        st = fg.sample_stats(seed=3)
        n = 100                                     # n_test = 97 rounded up to whole batches
        for i, f in enumerate(folds):
            s = st[i]
            assert s['n'] == n
            x = fg.generate(i, n, seed=3)
            pred, logits = fg.predict_rows(i, x)
            np.testing.assert_array_equal(s['counts'], np.bincount(pred, minlength=K))
            assert abs(s['score'][0] - _sig_lse(logits).mean()) <= 1e-6
            _, real_logits = fg.predict(i)
            assert abs(s['score'][1] - _sig_lse(real_logits).mean()) <= 1e-6
            assert s['mean'].shape == (2, 250) and s['cov'].shape == (2, 250, 250)
            np.testing.assert_array_equal(s['cov'], np.transpose(s['cov'], (0, 2, 1)))
            if precision != 'fp32':
                continue
            pD = [np.asarray(a, np.float64) for a in fg.get_params(i, 0)]
            resident = fg.debug_buffer(i, 51, NTE, f['D'])
            np.testing.assert_array_equal(resident, f['xte'])
            worst = 0.0
            for side, rows in ((0, x), (1, f['xte'])):
                feat, _ = O.disc_forward(pD, rows.astype(np.float64), upto_mid=True)
                for got, ref in ((s['mean'][side], feat.mean(axis=0)), (s['cov'][side], np.cov(feat, rowvar=False))):
                    worst = max(worst, np.abs(got - ref).max() / np.abs(ref).max())
            print("MEASURED stats fp32 fold %d %.3g" % (i, worst))
            assert worst <= 1e-5


def _copy_group(src, folds, idx, extra=None, precision='f16'):
    """A group of the folds idx of src (weights copied) plus optional extra folds (D, n_test), loaded with random rows."""
    shapes = [(folds[i]['D'], NTR, NTE, folds[i]['seed']) for i in idx] + [(D, NTR, nte, 77 + D) for D, nte in (extra or [])]
    fg = FoldGroup(shapes, model='gan', precision=precision, batch=B)
    for k, i in enumerate(idx):
        for net in (0, 1):
            fg.set_params(k, net, src.get_params(i, net))
        f = folds[i]
        fg.load_fold(k, f['xtr'], f['ytr'], f['xte'], f['yte'])
    rng = np.random.default_rng(3)
    for k, (D, nte) in enumerate(extra or [], start=len(idx)):
        fg.load_fold(k, rng.standard_normal((NTR, D)).astype(np.float32), (np.arange(NTR) % K).astype(np.int32),
                     rng.standard_normal((nte, D)).astype(np.float32), (np.arange(nte) % K).astype(np.int32))
    return fg


@pytest.mark.parametrize("precision", ["tf32", "f16"])
def test_stats_reproducible_and_grouping_independent(precision):
    """Repeated calls, a fold alone, and a group whose extra fold has 400 test rows (chunks of 400 rows instead of 150):
    the same bits, generated rows and statistics."""
    folds = _folds((400, 1200))
    n = 6 * B
    with _group('gan', precision, folds) as fg:
        ref = fg.sample_stats(n, seed=9)
        rows = [fg.generate(i, n, seed=9) for i in range(2)]
        again = fg.sample_stats(n, seed=9)
        with _copy_group(fg, folds, [1], precision=precision) as alone, \
                _copy_group(fg, folds, [0, 1], extra=[(640, 400)], precision=precision) as wide:
            for other, idx in ((again, [0, 1]), (alone.sample_stats(n, seed=9), [1]), (wide.sample_stats(n, seed=9), [0, 1])):
                for k, i in enumerate(idx):
                    for key in ('counts', 'score', 'mean', 'cov'):
                        assert other[k][key].tobytes() == ref[i][key].tobytes(), (i, key)
            assert alone.generate(0, n, seed=9).tobytes() == rows[1].tobytes()
            assert wide.generate(0, n, seed=9).tobytes() == rows[0].tobytes()


def test_no_side_effects():
    """Twin groups: one calls generate and sample_stats between epochs 1 and 2.  Epoch 2 and everything after it is bitwise
    the same, and so are the kernels launched per epoch."""
    folds = _folds((400, 1200))
    rng = np.random.default_rng(4)
    idx = [np.stack([rng.permutation(NTR) for _ in range(2)]).astype(np.int32) for _ in range(3)]

    def run(probe):
        out = []
        with _group('gan', 'f16', folds) as fg:
            if probe:
                fg.generate(1, 4 * B, seed=2)
                fg.sample_stats()
                fg.generate(0, B, z=np.ones((B, fg.noise_dim), np.float32))
            before = fg.kernel_launches
            out.append(fg.train_epoch(idx[0], idx[1], idx[2]))
            out.append(np.array([fg.kernel_launches - before]))
            for i in range(2):
                for net in (0, 1):
                    out += fg.get_params(i, net) + [a for m in fg.get_adam(i, net) for a in m]
                out.append(fg.fold_counters(i))
                out += [np.float32(fg.eval(i))] + list(fg.predict(i))
            out += fg.saliency()
        return out

    for a, b in zip(run(True), run(False)):
        np.testing.assert_array_equal(a, b)


def test_error_codes():
    ERR_ARG, ERR_STATE = -1, -4
    lib = _lib.load()
    folds = _folds((16, 16))
    x = np.zeros((4 * B, 16), np.float32)
    X = _lib.fptr(x)
    cnt, sc = np.zeros((2, K), np.int32), np.zeros((2, 2))
    mu, cv = np.zeros((2, 2, 250)), np.zeros((2, 2, 250, 250))
    stats = (_lib.iptr(cnt), _lib.dptr(sc), _lib.dptr(mu), _lib.dptr(cv))
    with FoldGroup([(16, NTR, NTE, 0)] * 2, batch=B) as fg:                        # GAN, not loaded
        h = fg._h
        assert lib.mrgan_sample_stats(h, B, 0, *stats) == ERR_STATE
        fg.set_params(0, 1, folds[0]['pG'])
        assert lib.mrgan_generate(h, 0, B, 0, None, X) == 0                        # parameters are enough
        assert lib.mrgan_generate(h, 0, B, 0, None, None) == ERR_ARG
        assert lib.mrgan_generate(h, 2, B, 0, None, X) == ERR_ARG
        assert lib.mrgan_generate(h, -1, B, 0, None, X) == ERR_ARG
        for n in (0, -B, B - 1, B + 1):
            assert lib.mrgan_generate(h, 0, n, 0, None, X) == ERR_ARG, n
            assert lib.mrgan_sample_stats(h, n, 0, *stats) == ERR_ARG, n
        assert lib.mrgan_sample_stats(h, B, 0, None, *stats[1:]) == ERR_ARG
        assert lib.mrgan_sample_stats(h, B, 0, *stats[:3], None) == ERR_ARG
        for i, f in enumerate(folds):
            fg.load_fold(i, f['xtr'], f['ytr'], f['xte'], f['yte'])
        assert lib.mrgan_sample_stats(h, 2 * B, 0, *stats) == 0
        with pytest.raises(ValueError):
            fg.generate(0, B, z=np.zeros((B, 99), np.float32))
    with _group('nn', 'fp32', folds[:1]) as fg:
        assert lib.mrgan_generate(fg._h, 0, 20, 0, None, X) == ERR_STATE
        assert lib.mrgan_sample_stats(fg._h, 20, 0, *stats) == ERR_STATE
        assert "GAN handle" in lib.mrgan_last_error(fg._h).decode()
    with FoldGroup([(16, NTR, NTE, 0)], model='svm') as fg:
        assert lib.mrgan_generate(fg._h, 0, B, 0, None, X) == ERR_STATE
        assert lib.mrgan_sample_stats(fg._h, B, 0, *stats) == ERR_STATE
    with FoldGroup([(16, NTR, NTE, 5)] * 2, batch=20) as fg:                      # virtual ranks
        fg.dp_init_virtual(2)
        for r in range(2):
            fg.set_params(r, 0, folds[0]['pD']); fg.set_params(r, 1, folds[0]['pG'])
            fg.load_fold(r, folds[0]['xtr'], folds[0]['ytr'], folds[0]['xte'], folds[0]['yte'])
        assert lib.mrgan_generate(fg._h, 0, 20, 0, None, X) == ERR_STATE
        assert lib.mrgan_sample_stats(fg._h, 20, 0, *stats) == ERR_STATE
        assert "data-parallel" in lib.mrgan_last_error(fg._h).decode()


def test_loaded_model_generates_the_live_rows(tmp_path):
    from test_gpu_checkpoint import _jobs
    job = _jobs()[1]
    path = str(tmp_path / 'model.npz')
    live = {}

    def on_epoch(epoch, fg, st, rngs):
        if epoch == 2:
            checkpoint.save(path, fg, 0, job, seed=3, epochs=2, epochs_done=2, perm='host', rng_state=rngs[0])
            live['x'] = fg.generate(0, 3 * fg.batch, seed=4)
            live['st'] = fg.sample_stats(seed=4)[0]

    mr_gan.train_gan_folds([job], epochs=2, seed=3, precision='f16', on_epoch=on_epoch)
    with checkpoint.load_model(path) as m:
        assert m.generate(0, 3 * m.batch, seed=4).tobytes() == live['x'].tobytes()
        st = m.sample_stats(seed=4)[0]
        for key in ('counts', 'score', 'mean', 'cov'):
            assert st[key].tobytes() == live['st'][key].tobytes(), key
        X = np.asarray(job['X'], np.float64)[job['test_idx']]
        np.testing.assert_allclose(m.inverse_transform(m.transform(X)), X, rtol=1e-5, atol=1e-5 * np.abs(X).max())


def _cli(argv, cwd):
    r = subprocess.run([sys.executable, '-c', 'import sys; sys.path.insert(0, %r); from mr_gan_b200 import mr_gan as m; '
                        'sys.exit(m.main(sys.argv[1:]))' % ROOT] + argv, capture_output=True, text=True, cwd=cwd, timeout=3000)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def test_cli_samples_and_rerun_from_checkpoints(tmp_path):
    base = ['--synthetic', '--tables', '6', '--epochs', '1', '--seed', '0', '--results']
    first = _cli(base + [str(tmp_path / 'r1.jsonl'), '--samples', str(tmp_path / 's1.npz'), '--checkpoint', str(tmp_path / 'ck')],
                 str(tmp_path))
    lines = [l for l in first.splitlines() if l.startswith('Samples: ')]
    assert len(lines) == 14 and first.count('Average error:') == 14
    with np.load(str(tmp_path / 's1.npz')) as z:
        index = json.loads(str(z['index']))
        assert sorted(k for k in z.files if k != 'index') == sorted('job_%d' % e['job_id'] for e in index)
        assert len(index) == 84 and all(np.isfinite(e['frechet']) and len(e['class_share']) == K for e in index)
        assert all(z['job_%d' % e['job_id']].shape[0] == 50 for e in index)
    recs = [json.loads(l) for l in open(str(tmp_path / 'r1.jsonl'))]
    assert len(recs) == 84 and all('fm_gap' in r and 'p_real_gen' in r for r in recs)
    rerun = _cli(base + [str(tmp_path / 'r2.jsonl'), '--samples', str(tmp_path / 's2.npz'), '--checkpoint', str(tmp_path / 'ck')],
                 str(tmp_path))
    assert rerun == first                                           # every job from its final checkpoint file
    assert open(str(tmp_path / 'r2.jsonl')).read() == open(str(tmp_path / 'r1.jsonl')).read()
    with np.load(str(tmp_path / 's1.npz')) as a, np.load(str(tmp_path / 's2.npz')) as b:
        assert sorted(a.files) == sorted(b.files) and all(a[k].tobytes() == b[k].tobytes() for k in a.files)
    plain = _cli(base[:-1], str(tmp_path))
    assert plain.splitlines() == [l for l in first.splitlines() if not l.startswith('Samples: ')]
