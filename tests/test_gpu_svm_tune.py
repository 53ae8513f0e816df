"""GPU tier of the SVM grid search (mrgan_svm_cv, mrgan_svm_fit_folds, mr_svm.py --tune): inner-CV error counts, the
selected point and the tuned test error against sklearn's GridSearchCV, reproducibility, grouping and grid independence,
the per-fold C refit against mrgan_svm_fit, error codes and the CLI."""
import ctypes
import json

import numpy as np
import pytest
from sklearn.model_selection import GridSearchCV, StratifiedKFold
from sklearn.svm import SVC

from mr_gan_b200 import _lib, foldprep, mr_svm, synthetic
from mr_gan_b200.engine import FoldGroup, MrganError
from mr_gan_b200.mr_gan import stack_objects

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


def _group(cases, fg=None):
    """cases: (modality, percent, loo).  A loaded SVM FoldGroup and per fold (FoldIndex, D)."""
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
    return fg, [(f, X.shape[1]) for X, y, f in folds]


def _cv(fg, folds, grid, cv):
    lab = np.stack([f.lab_rows for f, _ in folds])
    split = np.stack([mr_svm.inner_splits(f.y_train[f.lab_rows], cv) for f, _ in folds])
    D = np.array([d for _, d in folds], np.float64)
    gam = (np.array(grid['gamma_D'])[None, :] / D[:, None]).astype(np.float32)
    return lab, split, gam, fg.svm_cv(lab, split, grid['C'], gam)


# 1 % and 16 %: the default grid; 100 %: a smaller grid (sklearn's 100 inner fits of 4800 rows would take many CPU minutes)
TUNE_CASES = [((2, 1, False), mr_svm.DEFAULT_GRID, 5), ((2, 16, False), mr_svm.DEFAULT_GRID, 5),
              ((2, 100, False), dict(C=[1, 10], gamma_D=[0.5, 1]), 3), ((5, 16, True), mr_svm.DEFAULT_GRID, 5)]


@pytest.mark.parametrize("case,grid,cv", TUNE_CASES, ids=["m2-1pct", "m2-16pct", "m2-100pct", "m5-loo-16pct"])
def test_counts_selection_and_tuned_error_against_grid_search_cv(case, grid, cv):
    fg, folds = _group([case])
    try:
        lab, split, gam, wrong = _cv(fg, folds, grid, cv)
        (f, D), = folds
        ntr, nte = len(f.train_rows), len(f.test_rows)
        xl = fg.debug_buffer(0, 50, ntr, D)[f.lab_rows].astype(np.float64)
        xt = fg.debug_buffer(0, 51, nte, D).astype(np.float64)
        yl = f.y_train[f.lab_rows]
        nval = np.bincount(split[0], minlength=cv)
        mean, (ic, ig) = mr_svm.select(wrong[0], nval)
        # sklearn, with the float32 gamma the library uses
        gs = GridSearchCV(SVC(kernel='rbf', tol=1e-3), {'C': [float(c) for c in grid['C']], 'gamma': [float(g) for g in gam[0]]},
                          cv=StratifiedKFold(cv), n_jobs=-1).fit(xl, yl)
        nC, nG = len(grid['C']), len(grid['gamma_D'])
        acc = np.stack([gs.cv_results_['split%d_test_score' % s] for s in range(cv)], axis=1).reshape(nC, nG, cv)
        sk_wrong = np.rint((1.0 - acc) * nval).astype(np.int64).transpose(1, 0, 2)           # [nG, nC, cv]
        assert np.abs(wrong[0] - sk_wrong).max() <= 2, (wrong[0], sk_wrong)
        # the selected point: sklearn's, unless its lead is within what the count tolerance can move
        sk_mean = gs.cv_results_['mean_test_score'].reshape(nC, nG)
        tol = 2 * np.mean(2.0 / nval)
        order = np.sort(sk_mean.ravel())[::-1]
        if order[0] - order[1] > tol:
            assert (ic, ig) == divmod(gs.best_index_, nG)
        else:
            assert sk_mean[ic, ig] >= gs.best_score_ - tol
        # the refit with the selected point and the tuned test error
        fg.svm_fit(lab, C=[grid['C'][ic]], gamma=[gam[0, ig]])
        err = fg.svm_eval(0)
        if (ic, ig) == divmod(gs.best_index_, nG):
            assert abs(err * nte - np.sum(gs.predict(xt) != f.y_test)) <= 2
    finally:
        fg.close()


def test_counts_reproducible_and_independent_of_grouping_and_grid():
    grid = dict(C=[1, 10], gamma_D=[0.5, 2])
    fg, folds = _group([(2, 16, False)])
    _, _, _, alone = _cv(fg, folds, grid, 5)
    _, _, _, again = _cv(fg, folds, grid, 5)
    assert np.array_equal(alone, again)
    _, _, _, one_gamma = _cv(fg, folds, dict(C=grid['C'], gamma_D=[2]), 5)
    assert np.array_equal(one_gamma[:, 0], alone[:, 1])
    fg.close()
    fg, folds = _group([(5, 16, False), (2, 16, False)])        # another fold, another D, first in the group
    _, _, _, grouped = _cv(fg, folds, grid, 5)
    assert np.array_equal(grouped[1], alone[0])
    fg.close()


def test_fit_folds_with_broadcast_c_equals_svm_fit():
    fg, folds = _group([(2, 16, False), (5, 16, False)])
    try:
        lab = np.ascontiguousarray(np.stack([f.lab_rows for f, _ in folds]), np.int32)
        gam = np.array([1.0 / d for _, d in folds], np.float32)
        it = np.zeros((2, fg.n_pairs), np.int32)
        assert fg.lib.mrgan_svm_fit(fg._h, _lib.iptr(lab), lab.shape[1], ctypes.c_float(1.0), _lib.fptr(gam), ctypes.c_float(1e-3),
                                    _lib.iptr(it)) == 0
        ref = [fg.svm_decision(i) for i in range(2)]
        it2 = fg.svm_fit(lab, C=[1.0, 1.0], gamma=gam)
        assert np.array_equal(it, it2)
        assert all(np.array_equal(r, fg.svm_decision(i)) for i, r in enumerate(ref))
        # per-fold C: each fold as fitted alone with its C
        it3 = fg.svm_fit(lab, C=[10.0, 1.0], gamma=gam)
        dec0 = fg.svm_decision(0)
        assert np.array_equal(it3[1], it[1]) and np.array_equal(fg.svm_decision(1), ref[1])
        fg.svm_fit(lab, C=10.0, gamma=gam)
        assert np.array_equal(fg.svm_decision(0), dec0)
    finally:
        fg.close()


def _code(fn, *a, **k):
    with pytest.raises(MrganError) as e:
        fn(*a, **k)
    return int(str(e.value).split()[2].rstrip(':'))


def test_error_codes():
    ERR_ARG, ERR_STATE = -1, -4
    rng = np.random.default_rng(0)
    X = rng.standard_normal((130, 8)).astype(np.float32)
    ytr, yte = np.repeat(np.arange(6), 20)[:110].astype(np.int32), np.arange(20).astype(np.int32) % 6
    lab = np.arange(0, 110, 2, dtype=np.int32)[None, :]            # class-major: labels of ytr are sorted
    yl = ytr[lab[0]]
    split = mr_svm.inner_splits(yl, 3)[None, :]
    with FoldGroup([(8, 110, 20, 0)]) as gan:
        assert _code(gan.svm_cv, lab, split, [1.0], [0.1]) == ERR_STATE
    with FoldGroup([(8, 110, 20, 0)], model='svm') as fg:
        assert _code(fg.svm_cv, lab, split, [1.0], [0.1]) == ERR_STATE          # before the fold data is loaded
        fg.load_fold(0, X[:110], ytr, X[110:], yte)
        bad = split.copy(); bad[0, 4] = -1
        assert _code(fg.svm_cv, lab, bad, [1.0], [0.1]) == ERR_ARG              # split index outside [0, n_splits)
        assert _code(fg.svm_cv, lab, np.zeros_like(split), [1.0], [0.1]) == ERR_ARG   # n_splits = 1
        lacks = (yl == 0).astype(np.int32)[None, :]                            # split 1 holds all of class 0
        assert _code(fg.svm_cv, lab, lacks, [1.0], [0.1]) == ERR_ARG
        assert _code(fg.svm_cv, lab, split, [1.0, 0.0], [0.1]) == ERR_ARG
        assert _code(fg.svm_cv, lab, split, [1.0], [0.1, -1.0]) == ERR_ARG
        assert _code(fg.svm_cv, lab, split, [], [0.1]) == ERR_ARG
        assert _code(fg.svm_cv, lab, split, [1.0], np.zeros((1, 0), np.float32)) == ERR_ARG
        assert _code(fg.svm_cv, lab[:, ::-1].copy(), split, [1.0], [0.1]) == ERR_ARG   # not class-major
        assert _code(fg.svm_fit, lab, C=[0.0]) == ERR_ARG
        fg.svm_fit(lab)
        e = fg.svm_eval(0)
        assert _code(fg.svm_cv, lab, lacks, [1.0], [0.1]) == ERR_ARG
        assert fg.svm_eval(0) == e                                             # a rejected call leaves the fit valid
        w = fg.svm_cv(lab, split, [0.5, 2.0], [0.05, 0.1, 0.2])
        assert w.shape == (1, 3, 2, 3) and np.all((w >= 0) & (w <= np.bincount(split[0])[None, None, None, :]))
        for call in (lambda: fg.svm_eval(0), lambda: fg.svm_decision(0), lambda: fg.predict(0), fg.confusion,
                     lambda: fg.predict_rows(0, X[110:115]), lambda: fg.time_op("svm_smo", reps=1)):
            assert _code(call) == ERR_STATE                                    # the CV invalidated the fit
        fg.svm_fit(lab)
        assert fg.svm_eval(0) == e


def test_cli_table2_tune(capsys, tmp_path):
    path = tmp_path / 'r.jsonl'
    assert mr_svm.main(['--tables', '2', '--synthetic', '--seed', '0', '--tune', '--results', str(path)]) == 0
    out = capsys.readouterr().out.splitlines()
    avg = [i for i, line in enumerate(out) if line.startswith('Average error:')]
    sel = [i for i, line in enumerate(out) if line.startswith('Selected C:')]
    assert len(avg) == 14 and [i + 1 for i in avg] == sel
    for i in sel:
        c_part, g_part = out[i][len('Selected C: '):].split(' Selected gamma*D: ')
        assert len(c_part.split()) == len(g_part.split()) == 6
        assert {float(v) for v in c_part.split()} <= set(mr_svm.DEFAULT_GRID['C'])
        assert {float(v) for v in g_part.split()} <= set(mr_svm.DEFAULT_GRID['gamma_D'])
    recs = [json.loads(line) for line in path.read_text().splitlines()]
    assert len(recs) == 84
    for r in recs:
        acc = np.asarray(r['cv_accuracy'])
        assert acc.shape == (4, 5) and 0 <= r['error'] <= 1
        ic, ig = mr_svm.DEFAULT_GRID['C'].index(r['C']), mr_svm.DEFAULT_GRID['gamma_D'].index(r['gamma_D'])
        assert acc[ic, ig] == acc.max() and np.argmax(acc) == ic * 5 + ig
