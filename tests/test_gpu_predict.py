"""GPU tier of the predictions (mrgan_predict, mrgan_predict_rows, mrgan_confusion): consistency with the error of
eval / nn_evaluate / svm_eval, the oracle's phase-0 forward, sklearn's SVC, bitwise reproduction of the resident test set by
predict_rows, independence of the fold grouping and of a pending epoch, error codes, and the mr_nn CLI's flags."""
import json
import re

import numpy as np
import pytest
from sklearn.model_selection import StratifiedKFold
from sklearn.svm import SVC

from mr_gan_b200 import _lib, foldprep, mr_nn, synthetic
from mr_gan_b200.engine import FoldGroup, MrganError
from mr_gan_b200.model import init_disc, init_gen
from oracle import gan_oracle as O

pytestmark = pytest.mark.gpu

K = 6
NTR, NTE = 300, 97                    # n_test not a multiple of the batch: the ragged tail is predicted too


def _folds(Ds, seed=0):
    out = []
    for i, D in enumerate(Ds):
        rng = np.random.default_rng(seed + 17 * i)
        y = np.tile(np.arange(K), (NTR + NTE) // K + 1)[:NTR + NTE].astype(np.int32)
        rng.shuffle(y)
        X = (rng.standard_normal((K, D))[y] + 2.0 * rng.standard_normal((len(y), D))).astype(np.float32)
        out.append(dict(D=D, seed=1000 + seed + i, xtr=X[:NTR], ytr=y[:NTR], xte=X[NTR:], yte=y[NTR:], pD=init_disc(D, rng), pG=init_gen(D, rng),
                        idx=[np.stack([rng.permutation(NTR) for _ in range(3)]).astype(np.int32) for _ in range(2)]))
    return out


def _group(model, precision, folds, epochs=1):
    """A trained group: GAN epochs from fixed permutations, or NN epochs over all training rows."""
    fg = FoldGroup([(f['D'], NTR, NTE, f['seed']) for f in folds], model=model, precision=precision,
                   batch=50 if model == 'gan' else 20)
    for i, f in enumerate(folds):
        if model == 'gan':
            fg.set_params(i, 1, f['pG'])
        fg.set_params(i, 0, f['pD'])
        fg.load_fold(i, f['xtr'], f['ytr'], f['xte'], f['yte'])
    for e in range(epochs):
        if model == 'gan':
            fg.train_epoch(*[np.stack([f['idx'][e][s] for f in folds]) for s in range(3)])
        else:
            fg.nn_train_epoch(np.stack([f['idx'][e][0] for f in folds]))
    return fg


def _check_consistent(fg, model, folds):
    conf = fg.confusion()
    assert conf.shape == (len(folds), K, K) and conf.dtype == np.int32
    out = []
    for i, f in enumerate(folds):
        pred, scores = fg.predict(i)
        assert pred.shape == (NTE,) and scores.shape == (NTE, K)
        np.testing.assert_array_equal(pred, np.argmax(scores, axis=1))        # first maximal logit
        wrong = int(np.sum(pred != f['yte']))
        if model == 'gan':
            assert np.float32(wrong) / np.float32(NTE) == fg.eval(i)
        else:
            assert np.float32(1.0) - np.float32(wrong) / np.float32(NTE) == np.float32(fg.nn_evaluate(i)[1])
        np.testing.assert_array_equal(conf[i], np.bincount(f['yte'] * K + pred, minlength=K * K).reshape(K, K))
        np.testing.assert_array_equal(conf[i].sum(axis=1), np.bincount(f['yte'], minlength=K))
        out.append((pred, scores))
    return conf, out


def _check_rows(fg, i, D, pred, scores, n_scores):
    """predict_rows over the fold's own resident X_test reproduces predict bitwise for n = 1, odd, n_test, > n_test."""
    xt = fg.debug_buffer(i, 51, NTE, D)
    for n in (1, 7, NTE, NTE + 13):
        idx = np.arange(n) % NTE
        p, s = fg.predict_rows(i, xt[idx])
        assert p.shape == (n,) and s.shape == (n, n_scores)
        np.testing.assert_array_equal(p, pred[idx])
        np.testing.assert_array_equal(s, scores[idx])


LOGIT_TOL = {"fp32": 1e-5, "tf32": 5e-3, "f16": 5e-3}


@pytest.mark.parametrize("precision", ["fp32", "tf32", "f16"])
@pytest.mark.parametrize("model", ["gan", "nn"])
def test_predictions_consistent_with_errors_oracle_and_rows(model, precision):
    """Heterogeneous group (D = 400 and 1200) after one epoch.  The logits are those of the oracle's phase-0 forward with
    the weights read back, to LOGIT_TOL relative to the largest logit.  Measured maximum on a B200: 9.4e-7 in fp32
    (accumulation order only), 7.9e-4 in tf32 and 8.8e-4 in f16 (10-bit operand mantissas)."""
    folds = _folds((400, 1200))
    with _group(model, precision, folds) as fg:
        conf, res = _check_consistent(fg, model, folds)
        errs = [fg.eval(i) for i in range(2)]
        for i, f in enumerate(folds):
            want = O.disc_forward([p.astype(np.float64) for p in fg.get_params(i, 0)], f['xte'].astype(np.float64))[0]
            rel = np.abs(res[i][1] - want).max() / max(1.0, np.abs(want).max())
            assert rel <= LOGIT_TOL[precision], rel
            _check_rows(fg, i, f['D'], *res[i], K)
        # predicting new rows leaves every result on the resident test set unchanged
        assert [fg.eval(i) for i in range(2)] == errs
        np.testing.assert_array_equal(fg.confusion(), conf)
        for i in range(2):
            p, s = fg.predict(i)
            np.testing.assert_array_equal(p, res[i][0])
            np.testing.assert_array_equal(s, res[i][1])


def test_gan_f16_fold_alone_equals_fold_in_group_and_pending_epoch_is_unchanged():
    folds = _folds((400, 1200))
    with _group('gan', 'f16', folds, epochs=2) as fg:
        conf = fg.confusion()
        both = [fg.predict(i) for i in range(2)]
        ref = fg.epoch_result()
    for i in range(2):
        with _group('gan', 'f16', [folds[i]], epochs=2) as fg:
            p, s = fg.predict(0)
            np.testing.assert_array_equal(p, both[i][0])
            np.testing.assert_array_equal(s, both[i][1])
            np.testing.assert_array_equal(fg.confusion()[0], conf[i])
    # an epoch launched with wait=False, then confusion(), then epoch_result(): the same statistics and weights
    with _group('gan', 'f16', folds, epochs=1) as a, _group('gan', 'f16', folds, epochs=1) as b:
        idx = [np.stack([f['idx'][1][s] for f in folds]) for s in range(3)]
        a.train_epoch(*idx, wait=False)
        ca = a.confusion()
        sa = a.epoch_result()
        sb = b.train_epoch(*idx)
        np.testing.assert_array_equal(sa, sb)
        np.testing.assert_array_equal(sa, ref)
        np.testing.assert_array_equal(ca, b.confusion())
        for i in range(2):
            for x, y in zip(a.get_params(i, 0), b.get_params(i, 0)):
                np.testing.assert_array_equal(x, y)


# ---------------------------------------------------------------- SVM
_DATA = {}


def _svm_data(modality, loo):
    if (modality, loo) not in _DATA:
        if loo:
            from mr_gan_b200.mr_gan import stack_objects
            X, y, spans = stack_objects(synthetic.synthetic_dataset(modality, leaveObjectOut=True, seed=0))
            a, b = spans[next(iter(spans))]
            rows = np.arange(len(y))
            split = (np.concatenate([rows[:a], rows[b:]]), rows[a:b])
        else:
            X, y = synthetic.synthetic_dataset(modality, seed=0)
            split = next(StratifiedKFold(6, shuffle=True, random_state=0).split(X, y))
        _DATA[(modality, loo)] = (X, y, split)
    return _DATA[(modality, loo)]


def _svm_fit(cases, tol=1e-3):
    folds = []
    for modality, percent, loo in cases:
        X, y, (tr, te) = _svm_data(modality, loo)
        folds.append((X, y, foldprep.prepare_fold_indices(y, tr, te, percent, None, np.random.default_rng(7))))
    fg = FoldGroup([(X.shape[1], len(f.train_rows), len(f.test_rows), i) for i, (X, y, f) in enumerate(folds)], model='svm')
    slots = {}
    for i, (X, y, f) in enumerate(folds):
        if id(X) not in slots:
            slots[id(X)] = len(slots)
            fg.load_dataset(slots[id(X)], X, y)
        fg.prepare_fold(i, slots[id(X)], f.train_rows, f.test_rows)
    fg.svm_fit(np.stack([f.lab_rows for _, _, f in folds]), C=1.0, tol=tol)
    return fg, folds


def _vote(dec):
    votes = np.zeros((len(dec), K), np.int64)
    p = 0
    for a in range(K):
        for b in range(a + 1, K):
            votes[:, a] += dec[:, p] > 0
            votes[:, b] += dec[:, p] <= 0
            p += 1
    return np.argmax(votes, axis=1)                  # the first class with the most votes


SVM_CASES = [(2, 1, False), (2, 16, False), (2, 100, False), (5, 100, True)]


@pytest.mark.parametrize("case", SVM_CASES, ids=["m2-1pct", "m2-16pct", "m2-100pct", "m5-loo-100pct"])
def test_svm_predictions_against_decisions_and_sklearn(case):
    fg, ((X, y, f),) = _svm_fit([case])
    with fg:
        D, nte = X.shape[1], len(f.test_rows)
        pred, scores = fg.predict(0)
        np.testing.assert_array_equal(scores, fg.svm_decision(0))
        np.testing.assert_array_equal(pred, _vote(scores))
        assert np.float32(np.sum(pred != f.y_test)) / np.float32(nte) == np.float32(fg.svm_eval(0))
        conf = fg.confusion()
        np.testing.assert_array_equal(conf[0], np.bincount(f.y_test * K + pred, minlength=K * K).reshape(K, K))
        xl = fg.debug_buffer(0, 50, len(f.train_rows), D)[f.lab_rows].astype(np.float64)
        xt = fg.debug_buffer(0, 51, nte, D)
        c = SVC(kernel='rbf', C=1.0, gamma=1.0 / D, shrinking=False, tol=1e-3, decision_function_shape='ovo')
        c.fit(xl, f.y_train[f.lab_rows])
        assert np.sum(pred != c.predict(xt.astype(np.float64))) <= 2
        if case == (2, 16, False):
            err = fg.svm_eval(0)
            _check_rows(fg, 0, D, pred, scores, K * (K - 1) // 2)
            np.testing.assert_array_equal(fg.svm_decision(0), scores)      # the resident results are unchanged
            assert fg.svm_eval(0) == err
            np.testing.assert_array_equal(fg.confusion(), conf)
            np.testing.assert_array_equal(fg.predict(0)[0], pred)


def test_svm_rows_of_another_fold_against_sklearn_and_grouping_independence():
    """predict_rows on rows outside the fold's labeled and test sets (its unlabeled training rows) matches sklearn's
    decision_function to 1e-3 (both solvers at tol 1e-5); a fold predicted alone and inside a heterogeneous group gives
    bitwise identical results."""
    fg, folds = _svm_fit([(2, 16, False), (5, 16, False)], tol=1e-5)
    with fg:
        X, y, f = folds[0]
        D = X.shape[1]
        xtr = fg.debug_buffer(0, 50, len(f.train_rows), D)
        rows = xtr[np.setdiff1d(np.arange(len(f.train_rows)), f.lab_rows)[:500]]
        p, s = fg.predict_rows(0, rows)
        xl = xtr[f.lab_rows].astype(np.float64)
        c = SVC(kernel='rbf', C=1.0, gamma=1.0 / D, shrinking=False, tol=1e-5, decision_function_shape='ovo')
        c.fit(xl, f.y_train[f.lab_rows])
        assert np.abs(s - c.decision_function(rows.astype(np.float64))).max() <= 1e-3
        np.testing.assert_array_equal(p, _vote(s))
        grouped = [fg.predict(i) for i in range(2)]
        conf = fg.confusion()
    for i in range(2):
        alone, _ = _svm_fit([[(2, 16, False), (5, 16, False)][i]], tol=1e-5)
        with alone:
            pa, sa = alone.predict(0)
            np.testing.assert_array_equal(pa, grouped[i][0])
            np.testing.assert_array_equal(sa, grouped[i][1])
            np.testing.assert_array_equal(alone.confusion()[0], conf[i])


# ---------------------------------------------------------------- error codes
def test_error_codes():
    ERR_ARG, ERR_STATE = -1, -4
    lib = _lib.load()
    pred = np.zeros(NTE + 1, np.int32)
    x = np.zeros((NTE + 1, 16), np.float32)
    conf = np.zeros((2, K, K), np.int32)
    P, X, Cf = _lib.iptr(pred), _lib.fptr(x), _lib.iptr(conf)
    folds = _folds((16, 16))
    with FoldGroup([(16, NTR, NTE, 0)]) as fg:                          # a GAN fold that is not loaded
        h = fg._h
        assert lib.mrgan_predict(h, 0, P, None) == ERR_STATE
        assert lib.mrgan_predict_rows(h, 0, X, 1, P, None) == ERR_STATE
        assert lib.mrgan_confusion(h, Cf) == ERR_STATE
    with _group('nn', 'fp32', folds[:1]) as fg:
        h = fg._h
        assert lib.mrgan_predict(h, 0, None, None) == ERR_ARG
        assert lib.mrgan_predict_rows(h, 0, None, 1, P, None) == ERR_ARG
        assert lib.mrgan_predict_rows(h, 0, X, 1, None, None) == ERR_ARG
        assert lib.mrgan_confusion(h, None) == ERR_ARG
        assert lib.mrgan_predict(h, 1, P, None) == ERR_ARG and lib.mrgan_predict(h, -1, P, None) == ERR_ARG
        assert lib.mrgan_predict_rows(h, 1, X, 1, P, None) == ERR_ARG
        assert lib.mrgan_predict_rows(h, 0, X, 0, P, None) == ERR_ARG
        assert lib.mrgan_predict_rows(h, 0, X, NTE + 1, P, None) == ERR_ARG
        assert lib.mrgan_predict_rows(h, 0, X, NTE, P, None) == 0
        with pytest.raises(ValueError):
            fg.predict_rows(0, x[:, :15])
    with FoldGroup([(16, NTR, NTE, 0)], model='svm') as fg:             # an SVM handle before svm_fit
        fg.load_fold(0, folds[0]['xtr'], folds[0]['ytr'], folds[0]['xte'], folds[0]['yte'])
        for call in (lambda: fg.predict(0), lambda: fg.predict_rows(0, x[:3]), fg.confusion):
            with pytest.raises(MrganError, match="error -4"):
                call()
    with FoldGroup([(16, NTR, NTE, 5)] * 2, batch=20) as fg:           # virtual ranks (local batch: a multiple of 4)
        fg.dp_init_virtual(2)
        for r in range(2):
            fg.set_params(r, 0, folds[0]['pD']); fg.set_params(r, 1, folds[0]['pG'])
            fg.load_fold(r, folds[0]['xtr'], folds[0]['ytr'], folds[0]['xte'], folds[0]['yte'])
        assert lib.mrgan_predict(fg._h, 0, P, None) == ERR_STATE
        assert lib.mrgan_predict_rows(fg._h, 0, X, 1, P, None) == ERR_STATE
        assert lib.mrgan_confusion(fg._h, Cf) == ERR_STATE


# ---------------------------------------------------------------- the mr_nn CLI end to end
def test_mr_nn_cli_confusion_and_results(capsys, tmp_path):
    base = ['--tables', '2', '--synthetic', '--seed', '0', '--epochs', '1']
    assert mr_nn.main(base) == 0
    plain = capsys.readouterr().out.splitlines()
    path = tmp_path / 'nn.jsonl'
    assert mr_nn.main(base + ['--confusion', '--results', str(path)]) == 0
    flagged = capsys.readouterr().out.splitlines()
    it = iter(flagged)
    assert all(line in it for line in plain)                            # the flagless lines, unchanged and in order
    recs = [json.loads(line) for line in path.read_text().splitlines()]
    assert len(recs) == 84
    avg = [line for line in flagged if line.startswith('Average error:')]
    blocks = [i for i, line in enumerate(flagged) if line.startswith('Confusion matrix')]
    assert len(avg) == len(blocks) == 14
    for k in range(14):
        setting = recs[6 * k:6 * k + 6]
        assert len({(r['modality'], r['percentlabeled']) for r in setting}) == 1
        assert [r['fold'] for r in setting] == list(range(6))
        assert re.match(r'Average error: (\S+) ', avg[k]).group(1) == str(np.mean([r['error'] for r in setting]))
        b = blocks[k]
        total = sum(int(v) for line in flagged[b + 2:b + 2 + K] for v in line.split()[1:])
        assert total == sum(r['n_test'] for r in setting) == sum(np.sum(r['confusion']) for r in setting)
