"""CPU tier of the SVM: the NumPy restatement of libsvm's solver (oracle/svm_oracle.py) against sklearn's SVC, and the
mr_svm CLI's job list against mr_nn's."""
import numpy as np
import pytest
from sklearn.model_selection import StratifiedKFold
from sklearn.svm import SVC

from mr_gan_b200 import foldprep, mr_nn, mr_svm, sweep, synthetic
from oracle import svm_oracle


def _small_fold(percent):
    X, y = synthetic.synthetic_dataset(1, seed=3, pokes=20)          # modality 1: D = 400
    tr, te = next(StratifiedKFold(6, shuffle=True, random_state=0).split(X, y))
    f = foldprep.prepare_fold(None, None, percent, None, [X[tr], X[te], y[tr], y[te]], np.random.default_rng(0))
    return f.x_train[f.lab_rows], f.y_train[f.lab_rows], f.x_test


@pytest.mark.parametrize("percent", [1, 4])
@pytest.mark.parametrize("tol", [1e-3, 1e-5])
def test_oracle_matches_libsvm(percent, tol):
    xl, yl, xt = _small_fold(percent)
    D = xl.shape[1]
    r = svm_oracle.fit_predict(xl, yl, xt, 1.0 / D, C=1.0, eps=tol)
    c = SVC(kernel='rbf', C=1.0, gamma=1.0 / D, shrinking=False, tol=tol, decision_function_shape='ovo').fit(
        xl.astype(np.float64), yl)
    np.testing.assert_allclose(r['dec'], c.decision_function(xt.astype(np.float64)), rtol=0, atol=1e-6)
    np.testing.assert_array_equal(r['pred'], c.predict(xt.astype(np.float64)))
    np.testing.assert_array_equal(r['n_iter'], c.n_iter_)


def test_main_requires_tables():
    with pytest.raises(SystemExit):
        mr_svm.main([])


def _captured_jobs(main, monkeypatch):
    seen = []

    def fake(jobs, train_group, **kw):
        seen.append([dict(j) for j in jobs])
        return [0.0] * len(jobs)

    monkeypatch.setattr(sweep, 'run_sharded', fake)
    assert main(['--tables', '2', '4', '--synthetic', '--seed', '5']) == 0
    return [j for batch in seen for j in batch]


def test_job_list_matches_mr_nn(monkeypatch, capsys):
    nn = _captured_jobs(mr_nn.main, monkeypatch)
    out_nn = capsys.readouterr().out
    svm = _captured_jobs(mr_svm.main, monkeypatch)
    out_svm = capsys.readouterr().out
    assert out_svm == out_nn                                            # same table layout
    assert len(svm) == len(nn) == 2 * 7 * 6 + 2 * 5 * 72
    for a, b in zip(nn, svm):
        assert a['job_id'] == b['job_id'] and a['percentlabeled'] == b['percentlabeled']
        np.testing.assert_array_equal(a['train_idx'], b['train_idx'])
        np.testing.assert_array_equal(a['test_idx'], b['test_idx'])
    # labeled rows: mr_nn.train_nn_folds draws them from the job's (seed, job_id) stream first
    for a, f in zip(nn[::37], mr_svm.prepare_folds(svm[::37], 5)):
        rng = np.random.default_rng([5, a['job_id']])
        g = foldprep.prepare_fold_indices(a['y'], a['train_idx'], a['test_idx'], a['percentlabeled'], None, rng)
        np.testing.assert_array_equal(g.train_rows, f.train_rows)
        np.testing.assert_array_equal(g.lab_rows, f.lab_rows)
        assert np.all(np.diff(g.y_train[g.lab_rows]) >= 0)             # class-major
