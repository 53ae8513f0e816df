"""CPU suite: the --confusion / --results flags of the three CLIs with fake trainers (no GPU), and dict results through
the fold-sharded sweep at world size 2 over gloo."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from mr_gan_b200 import mr_gan, mr_nn, mr_svm, results, synthetic
from mr_gan_b200.model import MATERIALS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = len(MATERIALS)
BLOCK = 2 + K          # title, header and one line per material


def _fake(js, *a, details=False, **kw):
    """Deterministic results: every test row of a job is predicted as class (y + s) % K, s = job_id % 2, so the error is
    s and the confusion is a (shifted) diagonal."""
    out = []
    for j in js:
        y = np.asarray(j['y'])[j['test_idx']]
        s = j['job_id'] % 2
        conf = np.bincount(y * K + (y + s) % K, minlength=K * K).reshape(K, K).astype(np.int32)
        e = float(np.mean((y + s) % K != y))
        out.append(dict(error=e, confusion=conf) if details else e)
    return out


CLIS = [(mr_gan, 'train_gan_folds', ['3', '5', '6']), (mr_nn, 'train_nn_folds', ['2', '4']), (mr_svm, 'train_svm_folds', ['4'])]


def _strip_blocks(lines):
    out, i = [], 0
    while i < len(lines):
        if lines[i].startswith('Confusion matrix'):
            i += BLOCK
            continue
        out.append(lines[i])
        i += 1
    return out


@pytest.mark.parametrize("mod,fn,tables", CLIS, ids=[c[0].__name__.split('.')[-1] for c in CLIS])
def test_flags_add_blocks_and_records_only(mod, fn, tables, monkeypatch, capsys, tmp_path):
    monkeypatch.setattr(mod, fn, _fake)
    base = ['--tables'] + tables + ['--synthetic', '--seed', '0']
    assert mod.main(base) == 0
    plain = capsys.readouterr().out.splitlines()
    path = tmp_path / 'r.jsonl'
    assert mod.main(base + ['--confusion', '--results', str(path)]) == 0
    flagged = capsys.readouterr().out.splitlines()
    assert _strip_blocks(flagged) == plain
    recs = [json.loads(line) for line in path.read_text().splitlines()]
    tool = mod.__name__.split('.')[-1]
    # one record per fold-training, one block per setting (right after its average line)
    avg = [i for i, line in enumerate(flagged) if line.startswith('Average')]
    blocks = [i for i, line in enumerate(flagged) if line.startswith('Confusion matrix')]
    assert [i + 1 for i in avg] == blocks
    n_settings = len(avg)
    loo = {t for t in tables if t in ('3', '4')}
    want = sum({'3': 2 * 5 * 72, '4': 2 * 5 * 72, '2': 2 * 7 * 6, '5': 4 * 7 * 6, '6': 2 * 7 * 6}[t] for t in tables)
    assert len(recs) == want
    objects = list(synthetic.synthetic_dataset(2, leaveObjectOut=True, seed=0))
    seen_obj = []
    for r in recs:
        assert r['tool'] == tool and r['seed'] == 0 and str(r['table']) in tables
        assert r['modality'] in mr_gan.MODALITIES
        assert isinstance(r['job_id'], int) and isinstance(r['error'], float)
        conf = np.asarray(r['confusion'])
        assert conf.shape == (K, K) and conf.sum() == r['n_test']
        assert r['error'] == float(r['job_id'] % 2)
        assert ('precision' in r and r['epochs'] == 100) == (tool != 'mr_svm')
        assert ('percentunlabeled' in r) == (r['table'] == 6)
        assert ('time' in r) == (r['table'] == 5)
        if str(r['table']) in loo:
            assert 'fold' not in r
            seen_obj.append(r['object'])
        else:
            assert 'object' not in r and 0 <= r['fold'] < 6
    if loo:
        assert seen_obj[:len(objects)] == objects            # leave-one-object-out: the held-out objects in printed order
    assert n_settings > 0
    # each block sums the confusion of its setting's records
    totals = [sum(int(v) for line in flagged[b + 2:b + BLOCK] for v in line.split()[1:]) for b in blocks]
    assert sum(totals) == sum(r['n_test'] for r in recs)


def test_default_output_has_no_flag_side_effects(monkeypatch, capsys, tmp_path):
    """details=False unless a flag asks for it: the trainers see the reference's call."""
    seen = []

    def spy(js, *a, details=False, **kw):
        seen.append(details)
        return _fake(js, *a, details=details, **kw)

    monkeypatch.setattr(mr_nn, 'train_nn_folds', spy)
    mr_nn.main(['--tables', '2', '--synthetic', '--seed', '0'])
    assert seen and not any(seen)
    seen.clear()
    mr_nn.main(['--tables', '2', '--synthetic', '--seed', '0', '--results', str(tmp_path / 'x.jsonl')])
    assert seen and all(seen)
    assert 'Confusion matrix' not in capsys.readouterr().out


def test_confusion_block_layout():
    conf = np.arange(K * K).reshape(K, K)
    lines = results.confusion_lines(conf)
    assert len(lines) == BLOCK
    assert lines[1].split() == MATERIALS
    for name, row, line in zip(MATERIALS, conf, lines[2:]):
        assert line.split() == [name] + [str(v) for v in row]


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
    return [dict(error=j['D'] / 1e4, confusion=np.full((6, 6), j['D'] + rank, np.int32)) for j in js]
res = sweep.run_sharded(jobs, train_group, group_size=2, key=lambda j: j['n'], cost=lambda j: j['D'])
assert [r['error'] for r in res] == [j['D'] / 1e4 for j in jobs], res               # job order kept
assert [int(r['confusion'][0, 0]) // 10 * 10 for r in res] == [j['D'] for j in jobs]
assert {int(r['confusion'][0, 0]) %% 10 for r in res} == {0, 1}                     # both ranks did work
dist.barrier(); dist.destroy_process_group()
print("OK", rank)
"""


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_dict_results_through_run_sharded_world_size_2_gloo(tmp_path):
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
