"""CPU suite of the generator samples: the Frechet distance (results.frechet) against closed forms, and mr_gan.py --samples
through the recording fake group of test_host_orchestration.py (the printed line, the .npz index, the --results fields, and
unchanged output without the flag).  No GPU."""
import json

import numpy as np
import pytest

from mr_gan_b200 import results, synthetic
from mr_gan_b200.model import MATERIALS

from test_host_orchestration import FakeGroup, mg

W = 250


def _cov(rng, n_rows, w=W):
    a = rng.standard_normal((n_rows, w))
    return np.cov(a, rowvar=False), a.mean(axis=0)


def test_frechet_zero_for_identical_moments():
    rng = np.random.default_rng(0)
    c, m = _cov(rng, 600)
    assert abs(results.frechet(m, c, m, c)) <= 1e-10


def test_frechet_diagonal_closed_form_and_symmetry():
    rng = np.random.default_rng(1)
    m1, m2 = rng.standard_normal(W), rng.standard_normal(W)
    a, b = rng.uniform(0.1, 3.0, W), rng.uniform(0.1, 3.0, W)
    want = np.sum((m1 - m2) ** 2) + np.sum((np.sqrt(a) - np.sqrt(b)) ** 2)
    got = results.frechet(m1, np.diag(a), m2, np.diag(b))
    assert got == pytest.approx(want, rel=1e-10)
    c1, _ = _cov(rng, 400)
    c2, _ = _cov(rng, 500)
    assert results.frechet(m1, c1, m2, c2) == pytest.approx(results.frechet(m2, c2, m1, c1), rel=1e-8)


def test_frechet_rank_deficient_is_finite_and_real():
    rng = np.random.default_rng(2)
    c_real, m_real = _cov(rng, 97)                   # 97 real rows < 250 features
    c_gen, m_gen = _cov(rng, 1200)
    d = results.frechet(m_gen, c_gen, m_real, c_real)
    assert isinstance(d, float) and np.isfinite(d) and d > 0
    d = results.frechet(m_real, c_real, m_real, c_real)      # sqrtm of a singular product: zero to ~1e-7 of the trace
    assert isinstance(d, float) and abs(d) <= 1e-6 * np.trace(c_real)


def test_sample_report_fields():
    rng = np.random.default_rng(3)
    mean = rng.standard_normal((2, W))
    c, _ = _cov(rng, 300)
    st = dict(counts=np.array([5, 0, 3, 2, 0, 0], np.int32), score=np.array([0.25, 0.75]), mean=mean, cov=np.stack([c, c]))
    r = results.sample_report(st)
    assert r['fm_gap'] == pytest.approx(np.mean((mean[0] - mean[1]) ** 2))
    assert r['frechet'] == pytest.approx(np.sum((mean[0] - mean[1]) ** 2), rel=1e-6)
    assert (r['p_real_gen'], r['p_real_real']) == (0.25, 0.75)
    np.testing.assert_allclose(r['class_share'], [0.5, 0, 0.3, 0.2, 0, 0])


class SampleGroup(FakeGroup):
    """The recording fake group with the two sample entry points: fold f's moments are those of a shift by its key."""

    def sample_stats(self, n=None, seed=0):
        self.calls.append(("sample_stats", n, seed))
        out = []
        for D, _, _, key in self.shapes:
            s = (key % 7) / 10.0
            out.append(dict(counts=np.array([3, 1, 1, 0, 0, 0], np.int32), score=np.array([0.4, 0.9]),
                            mean=np.stack([np.full(W, s), np.zeros(W)]), cov=np.stack([np.eye(W), np.eye(W)])))
        return out

    def generate(self, fold, n, seed=0, z=None):
        self.calls.append(("generate", fold, n, seed))
        return np.zeros((n, self.shapes[fold][0]), np.float32)


@pytest.fixture
def sample_fake(monkeypatch):
    FakeGroup.instances.clear()
    monkeypatch.setattr(mg, "FoldGroup", SampleGroup)
    monkeypatch.setattr(mg, "dataset", lambda modalities=0, leaveObjectOut=False, seed=0, data_dir=None, **kw:
                        synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=4, seed=seed, leaveObjectOut=leaveObjectOut))
    return SampleGroup


def test_samples_flag_prints_lines_and_writes_index(sample_fake, capsys, tmp_path):
    path, rec = tmp_path / 's.npz', tmp_path / 'r.jsonl'
    assert mg.main(["--tables", "6", "--epochs", "1", "--seed", "3", "--samples", str(path), "--results", str(rec)]) == 0
    out = capsys.readouterr().out.splitlines()
    lines = [l for l in out if l.startswith('Samples: ')]
    assert len(lines) == 14
    for k, l in enumerate(out):                      # right after each setting's average line
        if l.startswith('Samples: '):
            assert out[k - 1].startswith('Average error:')
    groups = sample_fake.instances
    assert all(("sample_stats", None, 0) in g.calls for g in groups)
    keys = {int(s[3]) for g in groups for s in g.shapes}
    with np.load(str(path)) as z:
        index = json.loads(str(z['index']))
        names = [k for k in z.files if k != 'index']
        assert len(index) == 84 == len(names)
        assert sorted(names) == sorted('job_%d' % e['job_id'] for e in index)
        assert all(z[n].shape == (50, 10) and z[n].dtype == np.float32 for n in names)
    # the fake's moments: Frechet = 250 s^2 = 250 * FM gap per fold, s = (key % 7) / 10; the line holds the setting's means
    first = [e for e in index if e['percentunlabeled'] == 0 and e['modality'] == index[0]['modality']]
    assert len(first) == 6
    want = np.mean([e['frechet'] for e in first])
    assert all(e['frechet'] == pytest.approx(W * e['fm_gap']) for e in index) and keys
    assert lines[0] == ('Samples: Frechet %.1f FM gap %.4f D(real) generated 0.40 real 0.90 classes ' % (want, want / W) +
                        ' '.join('%s %.2f' % (n, v) for n, v in zip(MATERIALS, [0.6, 0.2, 0.2, 0, 0, 0])))
    recs = [json.loads(l) for l in open(str(rec))]
    assert len(recs) == 84 and all(set(r) >= {'frechet', 'fm_gap', 'p_real_gen', 'p_real_real', 'class_share'} for r in recs)


def test_no_samples_flag_leaves_output_unchanged(sample_fake, capsys, monkeypatch, tmp_path):
    argv = ["--tables", "6", "--epochs", "1", "--seed", "3", "--results", str(tmp_path / 'a.jsonl')]
    assert mg.main(argv) == 0
    with_fake = capsys.readouterr().out
    assert not any(c[0] in ("sample_stats", "generate") for g in sample_fake.instances for c in g.calls)
    monkeypatch.setattr(mg, "FoldGroup", FakeGroup)
    argv[-1] = str(tmp_path / 'b.jsonl')
    assert mg.main(argv) == 0
    assert capsys.readouterr().out == with_fake and 'Samples:' not in with_fake
    assert open(str(tmp_path / 'a.jsonl')).read() == open(str(tmp_path / 'b.jsonl')).read()


def test_nn_and_svm_have_no_samples_flag():
    from mr_gan_b200 import mr_nn, mr_svm
    for m in (mr_nn, mr_svm):
        with pytest.raises(SystemExit):
            m.main(['--tables', '4', '--synthetic', '--seed', '0', '--samples', 'x.npz'])
