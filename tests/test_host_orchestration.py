"""CPU suite, part 4: the drop-in's host orchestration (mr_gan_b200/mr_gan.py, mr_nn.py, mr_svm.py) against a recording
stand-in for the C-ABI handle -- order of calls, shapes, index streams, stdout format.  No GPU, no compute."""
import importlib

import numpy as np
import pytest

from mr_gan_b200 import foldprep, synthetic, tables

mg = importlib.import_module("mr_gan_b200.mr_gan")
mn = importlib.import_module("mr_gan_b200.mr_nn")
ms = importlib.import_module("mr_gan_b200.mr_svm")


class FakeGroup:
    instances = []

    def __init__(self, shapes, model="gan", precision="fp32", device=0, batch=None, **kw):
        self.shapes, self.model, self.precision, self.batch = list(shapes), model, precision, batch
        self.n_folds, self.n_train = len(self.shapes), self.shapes[0][1]
        self.calls, self.params, self.datasets, self.epochs, self.rows, self.lab = [], {}, {}, [], {}, []
        FakeGroup.instances.append(self)

    def set_params(self, fold, net, params):
        self.calls.append(("set_params", fold, net))
        self.params[(fold, net)] = [np.asarray(p).shape for p in params]

    def load_dataset(self, slot, x, y):
        self.calls.append(("load_dataset", slot))
        self.datasets[slot] = (np.asarray(x).shape, np.asarray(y).shape)

    def prepare_fold(self, fold, slot, train_rows, test_rows):
        self.calls.append(("prepare_fold", fold, slot))
        self.rows[fold] = (np.array(train_rows), np.array(test_rows))
        D, ntr, nte, _ = self.shapes[fold]
        assert len(train_rows) == ntr and len(test_rows) == nte and not set(train_rows) & set(test_rows)

    def load_fold(self, fold, xtr, ytr, xte, yte):
        self.calls.append(("load_fold", fold))
        D, ntr, nte, _ = self.shapes[fold]
        assert xtr.shape == (ntr, D) and xte.shape == (nte, D) and xtr.dtype == np.float32 and ytr.dtype == np.int32

    def train_epoch(self, a, b, c, wait=True):
        for idx in (a, b, c):
            assert idx.shape == (self.n_folds, self.n_train) and idx.dtype == np.int32 and idx.min() >= 0 and idx.max() < self.n_train
        self.epochs.append((a.copy(), b.copy(), c.copy()))
        self.calls.append(("train_epoch",))

    def set_epoch_rows(self, fold, lab_rows, unl_rows=None):      # device-side permutations (the CLI's default)
        assert 0 < len(lab_rows) <= self.n_train and (unl_rows is None or len(unl_rows) <= self.n_train)
        self.calls.append(("set_epoch_rows", fold, len(lab_rows), None if unl_rows is None else len(unl_rows)))

    def train_epoch_seeded(self, epoch, wait=True):
        assert sum(c[0] == "set_epoch_rows" for c in self.calls) == self.n_folds
        self.calls.append(("train_epoch_seeded", epoch))

    def epoch_result(self):
        return np.tile(np.array([[1.5, 0.7, 0.25, 0.01, 0.3]], np.float32), (self.n_folds, 1))

    def nn_train_epoch(self, idx, wait=True):
        assert idx.shape[0] == self.n_folds and idx.shape[1] % self.batch == 0
        self.epochs.append(idx.copy())

    def eval(self, fold):
        return np.float32(0.125)

    def nn_evaluate(self, fold):
        return np.float32(0.2), np.float32(0.75)

    def svm_fit(self, lab_rows, C=1.0, gamma=None):
        assert lab_rows.shape[0] == self.n_folds and len(np.broadcast_to(gamma, (self.n_folds,))) == self.n_folds
        self.lab.append(np.array(lab_rows))
        self.calls.append(("svm_fit",))
        return np.zeros((self.n_folds, 15), np.int32)

    def svm_cv(self, lab_rows, split, C_grid, gamma):
        assert split.shape == lab_rows.shape and gamma.shape[0] == self.n_folds
        self.lab.append(np.array(lab_rows))
        self.calls.append(("svm_cv",))
        wrong = np.zeros((self.n_folds, gamma.shape[1], len(C_grid), int(split.max()) + 1), np.int32)
        wrong[:, 0, 1] = 1                      # every point but (C_grid[1], gamma[0]) is perfect: C_grid[0] is chosen
        return wrong

    def svm_eval(self, fold):
        return 0.375

    def confusion(self):
        return np.ones((self.n_folds, 6, 6), np.int32)

    def close(self):
        self.calls.append(("close",))


@pytest.fixture
def fake(monkeypatch):
    FakeGroup.instances.clear()
    monkeypatch.setattr(mg, "FoldGroup", FakeGroup)
    monkeypatch.setattr(mn, "FoldGroup", FakeGroup)
    monkeypatch.setattr(ms, "FoldGroup", FakeGroup)
    return FakeGroup


def _small():
    return synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=20, seed=0)        # [1440, 10]: 1200 test rows fit


def test_mr_gan_single_fold_call_sequence_and_prints(fake, capsys):
    X, y = _small()
    err = mg.mr_gan(X, y, percentlabeled=1, epochs=3, verbose=True, seed=4)
    assert err == pytest.approx(0.125)
    g = fake.instances[0]
    assert g.model == "gan" and g.shapes[0][:3] == (10, 240, 1200) and g.batch == 50      # 200*6 held out (mr_gan.py:81,88)
    names = [c[0] for c in g.calls]
    assert names == ["set_params", "set_params", "load_fold"] + ["train_epoch"] * 3 + ["close"]
    assert g.calls[0][2] == 1 and g.calls[1][2] == 0                                    # generator built first (mr_gan.py:110)
    out = capsys.readouterr().out
    assert "Epochs: 3" in out and "Training batches per epoch: 4" in out and "Testing batches per epoch: 24" in out
    assert "Epoch 3, time = 0s, loss labeled = 1.5000, loss unlabeled = 0.7000, train error = 0.2500, test error = 0.3000" in out
    # labeled stream only contains the 10 labeled rows per class; unlabeled streams are permutations (mr_gan.py:189-194)
    il, iu, iu2 = g.epochs[0]
    assert len(set(il[0])) == 60 and sorted(iu[0]) == list(range(240)) and sorted(iu2[0]) == list(range(240))
    assert not (g.epochs[0][1] == g.epochs[1][1]).all()                                  # fresh permutations every epoch


def test_index_jobs_use_the_device_side_fold_preparation(fake):
    X, y = synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=5, seed=0)            # [360, 10]
    jobs = mg._kfold_jobs(X, y, 0, percentlabeled=0.5, percentunlabeled=1.0)
    errs = mg.train_gan_folds(jobs, epochs=2, seed=1, precision="tf32")
    assert errs == [pytest.approx(0.125)] * 6
    g = fake.instances[0]
    assert g.precision == "tf32" and g.n_folds == 6 and all(s[:3] == (10, 300, 60) for s in g.shapes)
    assert [c for c in g.calls if c[0] == "load_dataset"] == [("load_dataset", 0)]     # one upload for all six folds
    assert sum(c[0] == "prepare_fold" for c in g.calls) == 6 and not any(c[0] == "load_fold" for c in g.calls)
    il, iu, _ = g.epochs[0]
    # table-6 path: unlabeled streams are restricted to the first (labeled + unlabeled) rows per class (mr_gan.py:107,197-200)
    assert all(len(set(iu[f])) <= 6 * (5 + 10) for f in range(6)) and all(len(set(il[f])) == 30 for f in range(6))
    # seeds make the whole host side reproducible
    mg.train_gan_folds(jobs, epochs=2, seed=1, precision="tf32")
    for a, b in zip(g.epochs, fake.instances[1].epochs):
        for u, v in zip(a, b):
            np.testing.assert_array_equal(u, v)


def test_mr_nn_host_loop(fake):
    X, y = synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=5, seed=0)
    jobs = mg._kfold_jobs(X, y, 0, percentlabeled=2)                                     # 20 labeled rows per class
    errs = mn.train_nn_folds(jobs, epochs=3, seed=2)
    assert errs == [pytest.approx(0.25)] * 6                                             # 1 - accuracy (mr_nn.py:118)
    g = fake.instances[0]
    assert g.model == "nn" and g.batch == 20 and len(g.epochs) == 3 and g.epochs[0].shape == (6, 120)
    assert all(len(set(g.epochs[0][f])) == 120 for f in range(6))                        # model.fit shuffles the labeled rows
    with pytest.raises(ValueError, match="multiple of the batch size"):
        mn.train_nn_folds(mg._kfold_jobs(X, y, 0, percentlabeled=0.3), epochs=1, seed=2)  # 3 rows per class -> 18 rows


def test_gan_nn_and_svm_load_the_same_folds(fake):
    """One loader for the three trainers: the same jobs and seed give every group the same shapes and rows, and the SVM fits
    the NN's labeled rows.  Per fold, the GAN sets the generator, then the discriminator, then prepares the fold; the NN
    sets the discriminator; the SVM only prepares the fold."""
    X, y = synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=5, seed=0)
    jobs = tables.kfold_jobs(X, y, 0, percentlabeled=2)
    for i, j in enumerate(jobs):
        j['job_id'] = 7 + i
    assert mg.train_gan_folds(jobs, epochs=1, seed=3) == [pytest.approx(0.125)] * 6
    assert mn.train_nn_folds(jobs, epochs=1, seed=3) == [pytest.approx(0.25)] * 6
    assert ms.train_svm_folds(jobs, seed=3, details=True)[0]['confusion'].sum() == 36
    tuned = ms.train_svm_folds(jobs, seed=3, grid=dict(C=[0.5, 2.0], gamma_D=[1.0]), cv=3)
    assert [(r['error'], r['C'], r['gamma_D']) for r in tuned] == [(0.375, 0.5, 1.0)] * 6
    gan, nn, svm, svm_tuned = fake.instances
    assert [g.model for g in fake.instances] == ["gan", "nn", "svm", "svm"]
    for g in (nn, svm, svm_tuned):
        assert g.shapes == gan.shapes
        for f in range(6):
            for a, b in zip(g.rows[f], gan.rows[f]):
                np.testing.assert_array_equal(a, b)
    nn_lab = np.stack([np.unique(e) for e in nn.epochs[0]])          # the NN's epoch permutes its labeled rows
    for lab in svm.lab + svm_tuned.lab:                                 # the fit, and the tuned group's CV and refit
        np.testing.assert_array_equal(np.sort(lab, axis=1), nn_lab)
    per_fold = {"gan": [("set_params", 1), ("set_params", 0), ("prepare_fold",)], "nn": [("set_params", 0), ("prepare_fold",)],
                "svm": [("prepare_fold",)]}
    for g in fake.instances:
        steps = [c[:1] + c[2:] if c[0] == "set_params" else c[:1] for c in g.calls
                 if c[0] in ("set_params", "prepare_fold")]
        assert steps == per_fold[g.model] * 6
        folds = [c[1] for c in g.calls if c[0] in ("set_params", "prepare_fold")]
        assert folds == sorted(folds)                                    # fold by fold


def test_cli_prints_reference_strings(fake, capsys, monkeypatch):
    monkeypatch.setattr(mg, "dataset", lambda modalities=0, leaveObjectOut=False, seed=0, data_dir=None, **kw:
                        synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=4, seed=seed, leaveObjectOut=leaveObjectOut))
    assert mg.main(["--tables", "6", "--epochs", "1", "--seed", "3"]) == 0
    out = capsys.readouterr().out
    assert "Testing performance as quantity of unlabeled data increases" in out                      # mr_gan.py:322
    assert out.count("Percentage of training data unlabeled:") == 14 and out.count("Average error:") == 14
    assert "Test error: 0.125 Test accuracy: 0.875" in out                                            # mr_gan.py:338
    assert mg.main(["--tables", "3", "--epochs", "1", "--seed", "3"]) == 0
    out = capsys.readouterr().out
    assert out.count("Average leave-one-object-out error:") == 10 and "plastic_00 Test error: 0.125" in out   # mr_gan.py:280-282


def test_loo_and_kfold_jobs_reproduce_the_reference_splits():
    """mr_gan.py:264-282 (table 3): one fold per held-out object, train = every other object's rows in dictionary order,
    test = the object's rows; mr_gan.py:255-257 (tables 1/5/6): stratified 6-fold -> 6000/1200 rows at N=7200."""
    import itertools
    mg = importlib.import_module("mr_gan_b200.mr_gan")
    rng = np.random.default_rng(3)
    objects = {}
    for o in range(9):                       # 9 objects x 100 pokes (the reference has 72 x 100)
        objects["obj%d" % o] = {"x": rng.standard_normal((100, 7)).astype(np.float32), "y": np.full(100, o % 6)}
    jobs = mg._loo_jobs(objects, percentlabeled=16)
    assert len(jobs) == len(objects)
    for j, (name, data) in zip(jobs, objects.items()):
        # literal restatement of mr_gan.py:274-278
        Xtest = np.array(data["x"]); ytest = np.array(data["y"])
        Xtrain = np.array(list(itertools.chain.from_iterable([d["x"] for n, d in objects.items() if n != name])))
        ytrain = np.array(list(itertools.chain.from_iterable([d["y"] for n, d in objects.items() if n != name])))
        assert j["name"] == name and j["percentlabeled"] == 16
        np.testing.assert_array_equal(j["X"][j["train_idx"]], Xtrain)
        np.testing.assert_array_equal(j["y"][j["train_idx"]], ytrain)
        np.testing.assert_array_equal(j["X"][j["test_idx"]], Xtest)
        np.testing.assert_array_equal(j["y"][j["test_idx"]], ytest)
        assert mg.job_rows(j) == (800, 100) and mg.job_width(j) == 7

    X = rng.standard_normal((7200, 5)).astype(np.float32)
    y = np.repeat(np.arange(6), 1200)
    kj = mg._kfold_jobs(X, y, 11, percentlabeled=50)
    assert len(kj) == 6 and all(mg.job_rows(j) == (6000, 1200) for j in kj)
    seen = np.concatenate([j["test_idx"] for j in kj])
    assert np.array_equal(np.sort(seen), np.arange(7200))                  # every row is tested exactly once
    for j in kj:
        assert np.bincount(y[j["test_idx"]], minlength=6).tolist() == [200] * 6     # stratified (mr_gan.py:81: 200 per class)
        assert not np.intersect1d(j["train_idx"], j["test_idx"]).size
    again = mg._kfold_jobs(X, y, 11, percentlabeled=50)
    assert all(np.array_equal(a["test_idx"], b["test_idx"]) for a, b in zip(kj, again))       # seeded -> reproducible
