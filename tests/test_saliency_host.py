"""CPU suite of the input-gradient saliency: the float64 reference against central differences, the --saliency flag of the
GAN / NN CLIs with fake trainers (no GPU), and saliency dicts through the fold-sharded sweep at world size 2 over gloo."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from mr_gan_b200 import mr_gan, mr_nn, mr_svm, results, synthetic
from mr_gan_b200.model import MATERIALS, init_disc

import saliency_ref as R
from test_results_cli import _fake, _free_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = len(MATERIALS)


@pytest.mark.parametrize("alpha", [0.0, 0.3], ids=["relu", "leaky"])
@pytest.mark.parametrize("given", [False, True], ids=["predicted", "given"])
def test_reference_input_grad_matches_central_differences(alpha, given):
    rng = np.random.default_rng(3)
    D, n = 10, 4
    pD = [p.astype(np.float64) for p in init_disc(D, rng)]
    x = rng.standard_normal((n, D))
    t = rng.integers(0, K, n) if given else None
    g = R.input_grad(pD, x, t, alpha=alpha)
    assert g.shape == (n, D)
    tt = t if given else np.argmax(R.O.disc_forward(pD, x, None, alpha=alpha)[0], axis=1)
    eps = 1e-6
    fd = np.empty_like(x)
    for j in range(D):
        e = np.zeros(D)
        e[j] = eps
        fd[:, j] = (R.log_prob(pD, x + e, tt, alpha) - R.log_prob(pD, x - e, tt, alpha)) / (2 * eps)
    assert np.abs(g - fd).max() <= 1e-6 * np.abs(g).max()


def _fake_sal(js, *a, details=False, saliency=False, **kw):
    """_fake plus a deterministic profile per job: [K, D] filled with job_id + 1 + the feature index / D."""
    out = _fake(js, *a, details=details or saliency, **kw)
    if saliency:
        for j, r in zip(js, out):
            D = j['X'].shape[1]
            r['saliency'] = np.tile((j['job_id'] + 1 + np.arange(D) / D).astype(np.float32), (K, 1))
    return out


def test_saliency_flag_adds_share_lines_and_npz(monkeypatch, capsys, tmp_path):
    seen = []

    def spy(js, *a, **kw):
        seen.append(kw.get('saliency', False))
        return _fake_sal(js, *a, **kw)

    monkeypatch.setattr(mr_nn, 'train_nn_folds', spy)
    base = ['--tables', '2', '--synthetic', '--seed', '0']
    assert mr_nn.main(base) == 0
    plain = capsys.readouterr().out.splitlines()
    assert seen and not any(seen)                         # no flag: the trainers get saliency=False
    seen.clear()
    path = tmp_path / 's.npz'
    assert mr_nn.main(base + ['--confusion', '--saliency', str(path)]) == 0
    flagged = capsys.readouterr().out.splitlines()
    assert seen and all(seen)
    shares = [i for i, line in enumerate(flagged) if line.startswith('Saliency share:')]
    conf = [i for i, line in enumerate(flagged) if line.startswith('Confusion matrix')]
    assert [c + 2 + K for c in conf] == shares            # right after each setting's confusion block
    assert [line for i, line in enumerate(flagged) if i not in shares and not any(c <= i < c + 2 + K for c in conf)] == plain
    with np.load(str(path)) as z:
        index = json.loads(str(z['index']))
        arrays = {k: z[k] for k in z.files if k != 'index'}
    assert len(index) == len(arrays) == 2 * 7 * 6
    widths = {2: synthetic.feature_width(2), 5: synthetic.feature_width(5)}
    for rec in index:
        a = arrays['job_%d' % rec['job_id']]
        mod = mr_gan.MODALITIES.index(rec['modality'])
        assert rec['tool'] == 'mr_nn' and rec['table'] == 2 and 0 <= rec['fold'] < 6
        assert rec['blocks'] == [[n, w] for n, w in synthetic.block_widths(mod)]
        assert a.shape == (K, widths[mod]) and a.dtype == np.float32
    # each printed share line is the block mass of its setting's profiles, and sums to 1
    for s, i in enumerate(shares):
        recs = index[6 * s:6 * s + 6]
        blocks = recs[0]['blocks']
        want = results.block_shares([arrays['job_%d' % r['job_id']] for r in recs], blocks)
        assert abs(want.sum() - 1.0) < 1e-12
        got = flagged[i].split()[2:]
        assert got[0::2] == [b[0] for b in blocks]
        assert [float(v) for v in got[1::2]] == [float('%.3f' % v) for v in want]


def test_gan_cli_passes_saliency_with_blocks_of_table_5(monkeypatch, capsys, tmp_path):
    monkeypatch.setattr(mr_gan, 'train_gan_folds', _fake_sal)
    path = tmp_path / 'g.npz'
    assert mr_gan.main(['--tables', '5', '--synthetic', '--seed', '0', '--saliency', str(path)]) == 0
    out = capsys.readouterr().out.splitlines()
    assert sum(line.startswith('Saliency share:') for line in out) == 4 * 7
    with np.load(str(path)) as z:
        index = json.loads(str(z['index']))
        for rec in index:
            mod = mr_gan.MODALITIES.index(rec['modality'])
            kw = dict(contactmicTime=rec['time']) if mod == 3 else dict(forcetempTime=rec['time'])
            assert rec['blocks'] == [[n, w] for n, w in synthetic.block_widths(mod, **kw)]
            assert z['job_%d' % rec['job_id']].shape[1] == sum(w for _, w in rec['blocks'])


def test_svm_cli_has_no_saliency_flag():
    with pytest.raises(SystemExit):
        mr_svm.main(['--tables', '4', '--synthetic', '--seed', '0', '--saliency', 'x.npz'])


def test_share_line_format():
    blocks = [('temperature', 2), ('force0', 2), ('force1', 2)]
    prof = [np.array([[1.0, 1.0, 2.0, 0.0, 1.0, 1.0]]), np.array([[0.0, 0.0, 0.0, 2.0, 0.0, 0.0]])]
    sh = results.block_shares(prof, blocks)
    np.testing.assert_allclose(sh, [0.25, 0.5, 0.25])
    assert results.share_line(sh, blocks) == 'Saliency share: temperature 0.250 force0 0.500 force1 0.250'


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
    return [dict(error=j['D'] / 1e4, confusion=np.zeros((6, 6), np.int32),
                 saliency=np.full((6, j['D']), j['D'] + rank, np.float32)) for j in js]
res = sweep.run_sharded(jobs, train_group, group_size=2, key=lambda j: j['n'], cost=lambda j: j['D'])
assert [r['saliency'].shape for r in res] == [(6, j['D']) for j in jobs], res          # job order kept
assert [r['saliency'].dtype for r in res] == [np.float32] * len(jobs)
assert {int(r['saliency'][0, 0]) %% 10 for r in res} == {0, 1}                       # both ranks did work
dist.barrier(); dist.destroy_process_group()
print("OK", rank)
"""


def test_saliency_dicts_through_run_sharded_world_size_2_gloo(tmp_path):
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
