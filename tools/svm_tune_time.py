"""Cost of the SVM grid search (mr_svm.py --tune) on one table-2 setting: modality 2 (D = 1200), the 6 folds of one
percentage, the default grid (4 C x 5 gamma, 5 inner splits), at 1 %, 16 % and 100 % labeled.  For each percentage it
reports the wall time of FoldGroup.svm_cv (the call ends in a stream synchronise) and of the whole tuned fold-training
(train_svm_folds with grid: folds, CV, selection, refit, evaluation); on the 100 % group also time_op('svm_smo') of the refit.
The CPU arm is sklearn's GridSearchCV(SVC(kernel='rbf'), n_jobs=-1) on one 100 % fold, on this host's cores.  Prints one
JSON line per measurement, with the card's name and power limit.

    python tools/svm_tune_time.py [--percents 1 16 100] [--no-sklearn]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

from mr_gan_b200 import mr_svm  # noqa: E402
from mr_gan_b200.mr_gan import dataset  # noqa: E402
from mr_gan_b200.tables import kfold_jobs  # noqa: E402


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--percents', type=int, nargs='+', default=[1, 16, 100])
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--no-sklearn', action='store_true')
    a = ap.parse_args(argv)
    gpu, grid, cv = gpu_info(), mr_svm.DEFAULT_GRID, 5
    X, y = dataset(modalities=2, seed=a.seed, synthetic_data=True)
    for p in a.percents:
        jobs = kfold_jobs(X, y, a.seed + p, percentlabeled=p)
        for i, j in enumerate(jobs):
            j['job_id'] = i
        mr_svm.train_svm_folds(jobs, seed=a.seed, grid=grid, cv=cv)           # warm-up: module load, allocations
        fg, folds = mr_svm.load_group(jobs, seed=a.seed)
        try:
            lab = np.stack([f.lab_rows for f in folds])
            split = np.stack([mr_svm.inner_splits(f.y_train[f.lab_rows], cv) for f in folds])
            gam = np.array(grid['gamma_D'])[None, :] / np.array([s[0] for s in fg.shapes], np.float64)[:, None]
            t0 = time.perf_counter()
            fg.svm_cv(lab, split, grid['C'], gam)
            t_cv = time.perf_counter() - t0
        finally:
            fg.close()
        t0 = time.perf_counter()
        res = mr_svm.train_svm_folds(jobs, seed=a.seed, grid=grid, cv=cv)
        t_all = time.perf_counter() - t0
        rec = dict(op='svm_tune', percentlabeled=p, folds=len(jobs), n_lab=int(lab.shape[1]), grid=[len(grid['C']), len(grid['gamma_D'])],
                   cv=cv, svm_cv_s=round(t_cv, 3), tuned_training_s=round(t_all, 3),
                   selected_C=[r['C'] for r in res], selected_gamma_D=[r['gamma_D'] for r in res], gpu=gpu)
        if p == 100:                                                          # the SMO phase of the tuned refit
            fg, _ = mr_svm.tune_group(jobs, grid, cv, seed=a.seed)
            try:
                rec['svm_smo_ms'] = round(fg.time_op('svm_smo', reps=3), 3)
            finally:
                fg.close()
        print(json.dumps(rec), flush=True)
    if not a.no_sklearn and 100 in a.percents:
        from sklearn.model_selection import GridSearchCV, StratifiedKFold
        from sklearn.svm import SVC
        jobs = kfold_jobs(X, y, a.seed + 100, percentlabeled=100)
        f, = mr_svm.prepare_folds(jobs[:1], a.seed)
        tr = X[f.train_rows]
        mu, sd = tr.mean(0), tr.std(0)
        sd[sd == 0] = 1.0
        xl, yl = (tr[f.lab_rows] - mu) / sd, f.y_train[f.lab_rows]
        D = X.shape[1]
        gs = GridSearchCV(SVC(kernel='rbf', tol=1e-3), {'C': grid['C'], 'gamma': [g / D for g in grid['gamma_D']]},
                          cv=StratifiedKFold(cv), n_jobs=-1)
        t0 = time.perf_counter()
        gs.fit(xl, yl)
        t = time.perf_counter() - t0
        print(json.dumps(dict(op='sklearn_grid_search_cv', percentlabeled=100, folds=1, n_lab=len(yl), grid=[len(grid['C']), len(grid['gamma_D'])],
                              cv=cv, wall_s=round(t, 2), cpu_cores=os.cpu_count(), best=gs.best_params_, gpu=gpu)), flush=True)


if __name__ == '__main__':
    main()
