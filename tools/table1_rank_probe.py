"""One rank's share of the 8-GPU table-1 sweep on ONE GPU: trains the mixed-width group that sweep.plan deals to rank 0 for a
few epochs, times it, and checks that the same folds trained in one-modality groups give bit-identical errors."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from mr_gan_b200 import mr_gan as mg, sweep, tables

epochs = int(sys.argv[1]) if len(sys.argv) > 1 else 3
world = int(sys.argv[2]) if len(sys.argv) > 2 else 8
seed = 0
percents = [1, 2, 4, 8, 16, 50, 100]
jobs = []
for modality in range(len(tables.MODALITIES)):
    X, y = mg.dataset(modalities=modality, seed=seed, synthetic_data=True)
    jobs += [j for p in percents for j in tables.kfold_jobs(X, y, seed + p, percentlabeled=p)]
for i, j in enumerate(jobs):
    j['job_id'] = i
pl = sweep.plan(jobs, world, 42, key=tables.job_rows, cost=mg.job_cost)
g = pl[0][0]
print("rank 0 of %d: %d groups, first group %d folds, widths %s" % (world, len(pl[0]), len(g), [tables.job_width(jobs[i]) for i in g]))
mg.train_gan_folds([jobs[i] for i in g[:8]], epochs=1, seed=seed, precision='f16', device=0)      # library load, CUDA context
times = {}
for ep in (1, epochs):
    t0 = time.perf_counter()
    err = mg.train_gan_folds([jobs[i] for i in g], epochs=ep, seed=seed, precision='f16', device=0)
    times[ep] = time.perf_counter() - t0
    print("mixed group, %d epochs: %.2f s" % (ep, times[ep]))
per = (times[epochs] - times[1]) / max(epochs - 1, 1)
print("per epoch: %.3f s, set-up %.2f s -> 100 epochs ~ %.1f s" % (per, times[1] - per, times[1] + 99 * per))
# the same folds, grouped by modality
ref = {}
by_w = {}
for i in g:
    by_w.setdefault(tables.job_width(jobs[i]), []).append(i)
for w, idxs in by_w.items():
    for i, e in zip(idxs, mg.train_gan_folds([jobs[i] for i in idxs], epochs=epochs, seed=seed, precision='f16', device=0)):
        ref[i] = e
same = all(ref[i] == e for i, e in zip(g, err))
print("errors identical to one-modality groups:", same, "mean err", float(np.mean(err)))
sys.exit(0 if same else 1)
