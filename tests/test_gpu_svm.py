"""GPU tier of the SVM (MRGAN_MODEL_SVM, csrc/kernels_svm.cuh): kernel matrices against float64, the batched SMO
solver against sklearn's libsvm and against the NumPy restatement (oracle/svm_oracle.py), grouping independence,
reproducibility, error codes and the mr_svm CLI."""
import numpy as np
import pytest
from sklearn.model_selection import StratifiedKFold
from sklearn.svm import SVC

from mr_gan_b200 import foldprep, mr_svm, sweep, synthetic
from mr_gan_b200.engine import FoldGroup, MrganError
from mr_gan_b200.mr_gan import stack_objects
from oracle import svm_oracle

pytestmark = pytest.mark.gpu

_DATA = {}


def _data(modality, loo=False):
    if (modality, loo) not in _DATA:
        if loo:
            X, y, spans = stack_objects(synthetic.synthetic_dataset(modality, leaveObjectOut=True, seed=0))
            a, b = spans[next(iter(spans))]
            rows = np.arange(len(y))
            split = (np.concatenate([rows[:a], rows[b:]]), rows[a:b])
        else:
            X, y = synthetic.synthetic_dataset(modality, seed=0)
            split = next(StratifiedKFold(6, shuffle=True, random_state=0).split(X, y))
        _DATA[(modality, loo)] = (X, y, split)
    return _DATA[(modality, loo)]


def _fit(cases, tol=1e-3, fg=None):
    """cases: list of (modality, percent, loo).  Returns per fold dict(dec, err, iters, xl, yl, xt, yt, fi) and the group."""
    folds = []
    for modality, percent, loo in cases:
        X, y, (tr, te) = _data(modality, loo)
        folds.append((X, y, foldprep.prepare_fold_indices(y, tr, te, percent, None, np.random.default_rng(7))))
    if fg is None:
        fg = FoldGroup([(X.shape[1], len(f.train_rows), len(f.test_rows), i) for i, (X, y, f) in enumerate(folds)], model='svm')
    slots = {}
    for i, (X, y, f) in enumerate(folds):
        if id(X) not in slots:
            slots[id(X)] = len(slots)
            fg.load_dataset(slots[id(X)], X, y)
        fg.prepare_fold(i, slots[id(X)], f.train_rows, f.test_rows)
    it = fg.svm_fit(np.stack([f.lab_rows for _, _, f in folds]), C=1.0, tol=tol)
    out = []
    for i, (X, y, f) in enumerate(folds):
        D, ntr, nte = X.shape[1], len(f.train_rows), len(f.test_rows)
        xtr, xt = fg.debug_buffer(i, 50, ntr, D), fg.debug_buffer(i, 51, nte, D)
        out.append(dict(dec=fg.svm_decision(i), err=fg.svm_eval(i), iters=it[i], xl=xtr[f.lab_rows], yl=f.y_train[f.lab_rows],
                        xt=xt, yt=f.y_test, D=D))
    return out, fg


_SK = {}


def _sklearn(case, r, tol):
    key = case + (tol,)
    if key not in _SK:
        c = SVC(kernel='rbf', C=1.0, gamma=1.0 / r['D'], shrinking=False, tol=tol, decision_function_shape='ovo')
        c.fit(r['xl'].astype(np.float64), r['yl'])
        xt = r['xt'].astype(np.float64)
        _SK[key] = dict(dec=c.decision_function(xt), pred=c.predict(xt), iters=np.asarray(c.n_iter_))
    return _SK[key]


@pytest.mark.parametrize("D", [10, 1200, 3632])
def test_kernel_matrices_against_float64(D):
    rng = np.random.default_rng(D)
    if D == 10:
        X, y = rng.standard_normal((1300, D)), np.repeat(np.arange(6), [220, 215, 217, 216, 216, 216])
        tr, te = next(StratifiedKFold(6, shuffle=True, random_state=0).split(X, y))
        cases = None
    fg = None
    if D == 10:
        f = foldprep.prepare_fold_indices(y, tr, te, 16, None, np.random.default_rng(1))
        fg = FoldGroup([(D, len(tr), len(te), 0)], model='svm')
        fg.load_dataset(0, X, y)
        fg.prepare_fold(0, 0, f.train_rows, f.test_rows)
        fg.svm_fit(f.lab_rows[None, :])
        xl = fg.debug_buffer(0, 50, len(tr), D)[f.lab_rows]
        xt = fg.debug_buffer(0, 51, len(te), D)
    else:
        cases = [(2 if D == 1200 else 5, 16, False)]
        (r,), fg = _fit(cases)
        xl, xt = r['xl'], r['xt']
    g = float(np.float32(1.0 / D))
    n = len(xl)
    Kl, Kt = fg.debug_buffer(0, 60, n, n), fg.debug_buffer(0, 61, len(xt), n)
    fg.close()
    assert np.abs(Kl - svm_oracle.rbf(xl, xl, g)).max() <= 1e-6
    assert np.abs(Kt - svm_oracle.rbf(xt, xl, g)).max() <= 1e-6
    assert np.all(np.diag(Kl) == 1.0)


CASES = [(2, 1, False), (2, 16, False), (2, 100, False), (5, 100, True)]


@pytest.mark.parametrize("case", CASES, ids=["m2-1pct", "m2-16pct", "m2-100pct", "m5-loo-100pct"])
def test_solver_against_sklearn(case):
    (r5,), fg = _fit([case], tol=1e-5)
    fg.close()
    sk5 = _sklearn(case, r5, 1e-5)
    assert np.abs(r5['dec'] - sk5['dec']).max() <= 1e-3
    (r,), fg = _fit([case])
    fg.close()
    sk = _sklearn(case, r, 1e-3)
    n = len(r['yt'])
    votes = np.zeros((n, 6), np.int64)
    for p, (a, b) in enumerate(svm_oracle.pairs(6)):
        votes[:, a] += r['dec'][:, p] > 0
        votes[:, b] += r['dec'][:, p] <= 0
    pred = np.argmax(votes, axis=1)
    assert np.sum(pred == sk['pred']) >= n - 5
    assert abs(r['err'] * n - np.sum(sk['pred'] != r['yt'])) <= 2
    assert abs(r['err'] - np.mean(pred != r['yt'])) < 1e-6
    np.testing.assert_allclose(r['iters'], sk['iters'], rtol=0.10)


@pytest.mark.parametrize("case", CASES[:2], ids=["m2-1pct", "m2-16pct"])
def test_solver_against_oracle(case):
    (r,), fg = _fit([case])
    fg.close()
    o = svm_oracle.fit_predict(r['xl'], r['yl'], r['xt'], float(np.float32(1.0 / r['D'])), C=1.0, eps=1e-3)
    assert np.abs(r['dec'] - o['dec']).max() <= 1e-4
    np.testing.assert_allclose(r['iters'], o['n_iter'], rtol=0.10)


def test_grouping_independence_and_reproducibility():
    (alone,), fg = _fit([(2, 16, False)])
    fg.close()
    (a, b), fg = _fit([(2, 16, False), (5, 16, False)])          # different D, same n_train
    assert np.array_equal(alone['dec'], a['dec'])
    again, _ = _fit([(2, 16, False), (5, 16, False)], fg=fg)       # a second fit in the same handle
    assert np.array_equal(again[0]['dec'], a['dec']) and np.array_equal(again[1]['dec'], b['dec'])
    for op in ("svm_kmat", "svm_smo", "svm_predict"):               # re-running a phase reproduces it
        assert fg.time_op(op, reps=2) > 0
    assert np.array_equal(fg.svm_decision(1), b['dec'])
    fg.close()


def _code(fn, *a):
    with pytest.raises(MrganError) as e:
        fn(*a)
    return int(str(e.value).split()[2].rstrip(':'))


def test_error_codes():
    ERR_ARG, ERR_STATE = -1, -4
    rng = np.random.default_rng(0)
    X, y = rng.standard_normal((120, 8)).astype(np.float32), np.repeat(np.arange(6), 20).astype(np.int32)
    with FoldGroup([(8, 100, 20, 0)]) as gan:
        assert _code(gan.svm_fit, np.zeros((1, 12), np.int32)) == ERR_STATE
        assert _code(gan.svm_eval, 0) == ERR_STATE
        assert _code(gan.svm_decision, 0) == ERR_STATE
    with FoldGroup([(8, 100, 20, 0)], model='svm') as fg:
        lab = np.arange(0, 100, 5, dtype=np.int32)[None, :]
        assert _code(fg.svm_fit, lab) == ERR_STATE                   # before the fold data is loaded
        fg.load_fold(0, X[:100], np.repeat(np.arange(6), 17)[:100], X[100:], y[100:])
        assert _code(fg.eval, 0) == ERR_STATE
        assert _code(fg.nn_evaluate, 0) == ERR_STATE
        assert _code(fg.time_op, "dw1") == ERR_STATE
        assert _code(fg.train_batch_gen, 0, X[:50], np.zeros((50, 100), np.float32)) == ERR_STATE
        assert _code(fg.svm_eval, 0) == ERR_STATE                    # before svm_fit
        bad = lab.copy(); bad[0, 3] = 100
        assert _code(fg.svm_fit, bad) == ERR_ARG
        assert _code(fg.svm_fit, lab[:, ::-1].copy()) == ERR_ARG     # not class-major
        fg.svm_fit(lab)
        assert 0.0 <= fg.svm_eval(0) <= 1.0
    n = 8500
    yb = np.zeros(n + 10, np.int32); yb[4200:8400] = 1; yb[8400:] = np.arange(2, 6).repeat(28)[:n + 10 - 8400]
    with FoldGroup([(4, n + 10, 6, 0)], model='svm') as fg:
        fg.load_fold(0, rng.standard_normal((n + 10, 4)), yb, rng.standard_normal((6, 4)), np.arange(6))
        assert _code(fg.svm_fit, np.arange(n + 10, dtype=np.int32)[None, :]) == ERR_ARG   # pair (0, 1): 8400 rows


def test_cli_table2_against_sklearn(monkeypatch, capsys):
    got = {}
    real = sweep.run_sharded

    def spy(jobs, train_group, **kw):
        res = real(jobs, train_group, **kw)
        for j, e in zip(jobs, res):
            got[j['job_id']] = (j, e)
        return res

    monkeypatch.setattr(sweep, 'run_sharded', spy)
    assert mr_svm.main(['--tables', '2', '--synthetic', '--seed', '0']) == 0
    out = capsys.readouterr().out
    assert out.count('Average error:') == 14
    folds = [(j, e) for j, e in got.values() if j['X'].shape[1] == 1200 and j['percentlabeled'] == 16]
    assert len(folds) == 6
    for j, e in folds:
        f, = mr_svm.prepare_folds([j], 0)
        X, y = j['X'], j['y']
        tr = X[f.train_rows]
        mu, sd = tr.mean(0), tr.std(0)
        sd[sd == 0] = 1.0
        xl, xt = ((tr[f.lab_rows] - mu) / sd), ((X[f.test_rows] - mu) / sd)
        c = SVC(kernel='rbf', C=1.0, gamma=1.0 / X.shape[1]).fit(xl, f.y_train[f.lab_rows])
        assert abs(e * len(xt) - np.sum(c.predict(xt) != f.y_test)) <= 2
