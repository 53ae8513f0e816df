"""Measures mr_svm's tables 2 and 4 on synthetic data on one GPU and writes one JSON file (default
profiles/r03_svm_1gpu.json):

  - wall clock of the sweeps of ``mr_svm.py --tables 2 4 --synthetic`` (fold preparation, fit and prediction of every fold),
    run through the CLI itself with its stdout discarded;
  - device time per phase (kernel matrices, SMO, prediction) of every group, re-run once through mrgan_time_op;
  - achieved TFLOP/s of the kernel-matrix GEMM (3-term split: 3 x 2 x Kp per matrix element, from shapes) against the
    TF32 rate torch.mm measures on the same GPU in the same run;
  - SMO iterations per second per CTA (one CTA per fold and class pair);
  - the CPU arm: sklearn SVC on the same folds, one fold per host core, on a bounded SAMPLE of folds per labeled fraction,
    and GPU-vs-sklearn fold errors over the sampled folds.

    python tools/svm_bench.py [--out FILE] [--cpu-sample N]
"""
import argparse
import contextlib
import io
import json
import multiprocessing
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

from mr_gan_b200 import mr_svm, sweep  # noqa: E402
from mr_gan_b200.tables import job_rows  # noqa: E402


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'


def tf32_peak():
    import torch
    torch.backends.cuda.matmul.allow_tf32 = True
    a = torch.randn(8192, 8192, device='cuda')
    b = torch.randn(8192, 8192, device='cuda')
    for _ in range(3):
        torch.mm(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        torch.mm(a, b)
    e1.record()
    torch.cuda.synchronize()
    return 20 * 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12


_SAMPLE = []          # filled before the worker processes fork: the jobs' feature matrices are not pickled per task


def sk_fold(k):
    job, seed = _SAMPLE[k]
    X = job['X']
    from sklearn.svm import SVC
    f, = mr_svm.prepare_folds([job], seed)
    tr = X[f.train_rows]
    mu, sd = tr.mean(0), tr.std(0)
    sd[sd == 0] = 1.0
    xl, xt = (tr[f.lab_rows] - mu) / sd, (X[f.test_rows] - mu) / sd
    t = time.time()
    c = SVC(kernel='rbf', C=1.0, gamma=1.0 / X.shape[1]).fit(xl, f.y_train[f.lab_rows])
    err = float(np.mean(c.predict(xt) != f.y_test))
    return err, time.time() - t


def cli_sweeps(seed, group):
    """(jobs, errors, wall seconds) of every sweep mr_svm.py --tables 2 4 --synthetic runs, in its order."""
    runs, real = [], sweep.run_sharded

    def timed(jobs, train_group, **kw):
        t0 = time.time()
        errors = real(jobs, train_group, **kw)
        runs.append((jobs, errors, time.time() - t0))
        return errors

    sweep.run_sharded = timed
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            mr_svm.main(['--tables', '2', '4', '--synthetic', '--seed', str(seed), '--group', str(group)])
    finally:
        sweep.run_sharded = real
    return runs


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_svm_1gpu.json')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--group', type=int, default=42)
    ap.add_argument('--cpu-sample', type=int, default=2, help='sklearn folds per (table, modality, labeled %%)')
    args = ap.parse_args(argv)
    res = dict(gpu=gpu_info(), seed=args.seed, group=args.group)
    # 1. the sweeps as the CLI runs them
    runs = cli_sweeps(args.seed, args.group)
    jobs = [j for js, _, _ in runs for j in js]
    errors = [e for _, es, _ in runs for e in es]
    res['wall_s_tables_2_4'] = sum(t for *_, t in runs)
    res['folds'] = len(jobs)
    groups = sweep.plan(jobs, 1, args.group, key=lambda j: job_rows(j) + (j['percentlabeled'],))[0]
    # 2. per-phase device time of every group
    ph = dict(kmat_ms=0.0, smo_ms=0.0, predict_ms=0.0)
    flops, iters, ctas, smo_by_pct = 0.0, 0, 0, {}
    for idxs in groups:
        js = [jobs[i] for i in idxs]
        fg, it = mr_svm.fit_group(js, seed=args.seed)
        try:
            k, s, p = fg.time_op('svm_kmat', 1), fg.time_op('svm_smo', 1), fg.time_op('svm_predict', 1)
        finally:
            fg.close()
        ph['kmat_ms'] += k; ph['smo_ms'] += s; ph['predict_ms'] += p
        for j in js:
            D, (ntr, nte), n_lab = j['X'].shape[1], job_rows(j), 60 * j['percentlabeled']
            flops += 3 * 2 * ((D + 31) // 32 * 32) * (n_lab * n_lab + nte * n_lab)
        iters += int(it.sum()); ctas += it.size
        d = smo_by_pct.setdefault(js[0]['percentlabeled'], [0.0, 0, 0])
        d[0] += s; d[1] += int(it.sum()); d[2] += it.size
    res['device_ms'] = ph
    res['kmat_gemm_tflops'] = flops / (ph['kmat_ms'] * 1e-3) / 1e12
    res['tf32_peak_tflops_measured_torch_mm_8192'] = tf32_peak()
    res['kmat_fraction_of_measured_peak'] = res['kmat_gemm_tflops'] / res['tf32_peak_tflops_measured_torch_mm_8192']
    res['smo_iterations_total'] = iters
    res['smo_ctas'] = ctas
    res['smo_iters_per_s_per_cta'] = {str(p): (v[1] / v[2]) / (v[0] * 1e-3) for p, v in sorted(smo_by_pct.items())}
    # 3. CPU arm on a labelled sample
    sample = []
    for js, _, _ in runs:                       # one sweep per (table, modality); D names the modality
        t, D = '4' if 'name' in js[0] else '2', js[0]['X'].shape[1]
        for p in sorted({j['percentlabeled'] for j in js}):
            sel = [j for j in js if j['percentlabeled'] == p][:args.cpu_sample]
            sample += [(t, D, p, j) for j in sel]
    ncpu = os.cpu_count() or 1
    t0 = time.time()
    _SAMPLE[:] = [(j, args.seed) for *_, j in sample]
    with ProcessPoolExecutor(ncpu, mp_context=multiprocessing.get_context('fork')) as ex:
        out = list(ex.map(sk_fold, range(len(sample))))
    res['cpu_arm'] = dict(sample='%d folds per (table, modality, labeled %%)' % args.cpu_sample, host_cores=ncpu,
                          sample_folds=len(sample), sample_wall_s=time.time() - t0,
                          per_fold_s={'%s/D%d/%d%%' % (t, D, p): [] for t, D, p, _ in sample})
    by_id = {j['job_id']: e for j, e in zip(jobs, errors)}
    diffs = []
    for (t, D, p, j), (e, s) in zip(sample, out):
        res['cpu_arm']['per_fold_s']['%s/D%d/%d%%' % (t, D, p)].append(s)
        diffs.append(dict(table=t, D=D, percent=p, job_id=j['job_id'], gpu_err=by_id[j['job_id']], sklearn_err=e))
    res['errors_gpu_vs_sklearn'] = diffs
    res['mean_error_difference'] = float(np.mean([d['gpu_err'] - d['sklearn_err'] for d in diffs]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k not in ('errors_gpu_vs_sklearn', 'cpu_arm')}))
    return 0


if __name__ == '__main__':
    sys.exit(main())
