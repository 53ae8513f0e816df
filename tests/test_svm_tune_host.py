"""CPU suite of the SVM grid search (mr_svm.py --tune): the host-side selection against sklearn's GridSearchCV, the inner
splits against StratifiedKFold, the CLI flags with fake trainers, and tuned dicts through the fold-sharded sweep over gloo."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
from sklearn.model_selection import GridSearchCV, StratifiedKFold
from sklearn.svm import SVC

from mr_gan_b200 import mr_svm
from mr_gan_b200.model import MATERIALS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = len(MATERIALS)


def _data(seed=0, per_class=(9, 8, 10, 9, 11, 8), D=5):
    rng = np.random.default_rng(seed)
    y = np.repeat(np.arange(len(per_class)), per_class)                 # class-major, as svm_fit takes the labeled rows
    X = rng.standard_normal((len(y), D)) + 0.8 * y[:, None] * rng.standard_normal(D)[None, :]
    return X, y


def _counts(X, y, split, Cs, gammas):
    """wrong [nG, nC, n_splits] from sklearn SVC fits on the inner splits (the layout of FoldGroup.svm_cv)."""
    ns = int(split.max()) + 1
    w = np.zeros((len(gammas), len(Cs), ns), np.int64)
    for ig, g in enumerate(gammas):
        for ic, c in enumerate(Cs):
            for s in range(ns):
                tr, va = split != s, split == s
                pred = SVC(kernel='rbf', C=c, gamma=g, tol=1e-3).fit(X[tr], y[tr]).predict(X[va])
                w[ig, ic, s] = np.sum(pred != y[va])
    return w


def _check_against_grid_search(X, y, Cs, gammas, cv):
    split = mr_svm.inner_splits(y, cv)
    mean, (ic, ig) = mr_svm.select(_counts(X, y, split, Cs, gammas), np.bincount(split, minlength=cv))
    gs = GridSearchCV(SVC(kernel='rbf', tol=1e-3), {'C': Cs, 'gamma': gammas}, cv=StratifiedKFold(cv)).fit(X, y)
    assert np.array_equal(mean.ravel(), gs.cv_results_['mean_test_score'])        # bitwise
    assert gs.best_index_ == ic * len(gammas) + ig
    assert gs.best_params_ == {'C': Cs[ic], 'gamma': gammas[ig]}
    assert gs.best_score_ == mean[ic, ig]
    return mean, (ic, ig)


@pytest.mark.parametrize("cv", [3, 5])
def test_select_matches_grid_search_cv(cv):
    X, y = _data()
    _check_against_grid_search(X, y, [0.1, 1.0, 10.0], [0.05, 0.2, 1.0], cv)


def test_select_keeps_the_first_point_under_a_tie():
    X, y = _data(seed=1)
    mean, (ic, ig) = _check_against_grid_search(X, y, [1.0, 1.0, 10.0], [0.2, 0.2], 3)
    assert mean[0, 0] == mean[0, 1] == mean[1, 0] == mean[1, 1]
    assert (ic, ig) in ((0, 0), (2, 0))                                  # never a repeat of an earlier point
    # a synthetic all-equal grid: the first point wins
    w = np.full((3, 4, 5), 2)
    mean, best = mr_svm.select(w, np.full(5, 12))
    assert best == (0, 0) and np.all(mean == mean[0, 0])
    w[1, 2, :] = 1                                                       # a strictly better later point wins
    assert mr_svm.select(w, np.full(5, 12))[1] == (2, 1)


@pytest.mark.parametrize("per_class,cv", [((10, 10, 10, 10, 10, 10), 5), ((7, 12, 5, 9, 30, 6), 5), ((3, 4, 3, 5, 3, 3), 3)])
def test_inner_splits_are_stratified_kfold(per_class, cv):
    y = np.repeat(np.arange(len(per_class)), per_class)
    split = mr_svm.inner_splits(y, cv)
    assert split.dtype == np.int32 and split.shape == y.shape
    for s, (_, val) in enumerate(StratifiedKFold(cv).split(np.zeros((len(y), 1)), y)):
        assert np.array_equal(np.nonzero(split == s)[0], val)


def test_inner_splits_reject_more_splits_than_the_smallest_class():
    y = np.repeat(np.arange(6), [5, 5, 4, 5, 5, 5])
    with pytest.raises(ValueError):
        mr_svm.inner_splits(y, 5)
    mr_svm.inner_splits(y, 4)


def _fake(js, *a, details=False, grid=None, cv=5, **kw):
    """Deterministic trainer results: error job_id % 2; tuned, C and gamma_D are picked by job_id from the grid."""
    out = []
    for j in js:
        y = np.asarray(j['y'])[j['test_idx']]
        s = j['job_id'] % 2
        conf = np.bincount(y * K + (y + s) % K, minlength=K * K).reshape(K, K).astype(np.int32)
        r = dict(error=float(s), confusion=conf) if details else float(s)
        if grid is not None:
            r = r if isinstance(r, dict) else dict(error=r)
            nC, nG = len(grid['C']), len(grid['gamma_D'])
            r.update(C=grid['C'][j['job_id'] % nC], gamma_D=grid['gamma_D'][j['job_id'] % nG],
                     cv_accuracy=np.arange(nC * nG, dtype=np.float64).reshape(nC, nG) / 100 + cv)
        out.append(r)
    return out


def test_cli_tune_lines_and_records(monkeypatch, capsys, tmp_path):
    calls = []

    def spy(js, *a, **kw):
        calls.append((kw.get('grid'), kw.get('cv')))
        return _fake(js, *a, **kw)

    monkeypatch.setattr(mr_svm, 'train_svm_folds', spy)
    base = ['--tables', '2', '4', '--synthetic', '--seed', '0']
    assert mr_svm.main(base) == 0
    plain = capsys.readouterr().out.splitlines()
    assert calls and all(g is None for g, _ in calls)                    # no flag: the reference's fits only
    assert not any(line.startswith('Selected') for line in plain)
    calls.clear()
    path = tmp_path / 'r.jsonl'
    grid = dict(C=[0.5, 2.0, 8.0], gamma_D=[0.25, 1.0])
    assert mr_svm.main(base + ['--tune', '--C-grid', '0.5', '2', '8', '--gamma-grid', '0.25', '1', '--cv', '3',
                               '--confusion', '--results', str(path)]) == 0
    tuned = capsys.readouterr().out.splitlines()
    assert calls and all(g == grid and cv == 3 for g, cv in calls)
    sel = [i for i, line in enumerate(tuned) if line.startswith('Selected C:')]
    conf = [i for i, line in enumerate(tuned) if line.startswith('Confusion matrix')]
    assert [c + 2 + K for c in conf] == sel                              # right after each setting's confusion block
    assert [line for i, line in enumerate(tuned) if i not in sel and not any(c <= i < c + 2 + K for c in conf)] == plain
    recs = [json.loads(line) for line in path.read_text().splitlines()]
    assert len(recs) == 2 * 7 * 6 + 2 * 5 * 72
    by_setting, k = [], 0
    for i in sel:                                                        # the records of each setting, in printed order
        n = len(tuned[i].split('Selected gamma*D:')[1].split())
        by_setting.append(recs[k:k + n])
        k += n
    assert k == len(recs)
    for i, rs in zip(sel, by_setting):
        c_part, g_part = tuned[i][len('Selected C: '):].split(' Selected gamma*D: ')
        assert c_part.split() == ['%g' % r['C'] for r in rs]
        assert g_part.split() == ['%g' % r['gamma_D'] for r in rs]
        for r in rs:
            assert r['C'] == grid['C'][r['job_id'] % 3] and r['gamma_D'] == grid['gamma_D'][r['job_id'] % 2]
            assert np.array_equal(r['cv_accuracy'], np.arange(6).reshape(3, 2) / 100 + 3)
    assert tuned[sel[0]] == 'Selected C: 0.5 2 8 0.5 2 8 Selected gamma*D: 0.25 1 0.25 1 0.25 1'


def test_cli_tune_default_grid(monkeypatch, capsys):
    seen = []

    def spy(js, *a, **kw):
        seen.append(kw.get('grid'))
        return _fake(js, *a, **kw)

    monkeypatch.setattr(mr_svm, 'train_svm_folds', spy)
    assert mr_svm.main(['--tables', '2', '--synthetic', '--seed', '0', '--tune']) == 0
    out = capsys.readouterr().out.splitlines()
    assert seen and all(g == mr_svm.DEFAULT_GRID for g in seen)
    avg = [i for i, line in enumerate(out) if line.startswith('Average')]
    assert [i + 1 for i in avg] == [i for i, line in enumerate(out) if line.startswith('Selected C:')]
    assert 1 in mr_svm.DEFAULT_GRID['C'] and 1 in mr_svm.DEFAULT_GRID['gamma_D']   # the reference's point


WORKER = r"""
import os, sys
sys.path.insert(0, %r)
import numpy as np
import torch.distributed as dist
from mr_gan_b200 import sweep
dist.init_process_group("gloo")
rank = dist.get_rank()
jobs = [dict(D=d, n=6000 if i < 5 else 7100) for i, d in enumerate([400, 800, 1200] * 3)]
def train_group(js, dev):
    return [dict(error=j['D'] / 1e4, C=float(j['D'] + rank), gamma_D=0.5,
                 cv_accuracy=np.full((4, 5), j['D'] / 1e4, np.float64)) for j in js]
res = sweep.run_sharded(jobs, train_group, group_size=2, key=lambda j: j['n'], cost=lambda j: j['D'])
assert [r['error'] for r in res] == [j['D'] / 1e4 for j in jobs], res               # job order kept
assert [int(r['C']) // 10 * 10 for r in res] == [j['D'] for j in jobs]
assert all(r['cv_accuracy'].shape == (4, 5) and r['cv_accuracy'].dtype == np.float64 for r in res)
assert all(r['cv_accuracy'][0, 0] == j['D'] / 1e4 and r['gamma_D'] == 0.5 for r, j in zip(res, jobs))
assert {int(r['C']) %% 10 for r in res} == {0, 1}                                   # both ranks did work
dist.barrier(); dist.destroy_process_group()
print("OK", rank)
"""


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_tuned_dicts_through_run_sharded_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    port = _free_port()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, o
        assert ("OK %d" % r) in o, o
