"""Device time of mrgan_sample_stats's pass on a table-1 group: 42 GAN folds of D = 1200 (force + temperature), n_train =
6000, n_test = 1200, through mrgan_time_op: per fold 1200 generated rows (G's forward, BatchNorm per batch, D's eval forward,
statistics) and the 1200 resident test rows (D's eval forward, statistics).  Prints one JSON line with the card's name and
power limit.

    python tools/sample_time.py [--precision f16] [--folds 42] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

from mr_gan_b200.engine import FoldGroup  # noqa: E402
from mr_gan_b200.model import init_disc, init_gen  # noqa: E402


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--precision', default='f16', choices=['fp32', 'tf32', 'f16'])
    ap.add_argument('--folds', type=int, default=42)
    ap.add_argument('--reps', type=int, default=20)
    a = ap.parse_args()
    D, ntr, nte, K = 1200, 6000, 1200, 6
    rng = np.random.default_rng(0)
    with FoldGroup([(D, ntr, nte, i) for i in range(a.folds)], model='gan', precision=a.precision) as fg:
        for i in range(a.folds):
            fg.set_params(i, 0, init_disc(D, rng))
            fg.set_params(i, 1, init_gen(D, rng))
            fg.load_fold(i, rng.standard_normal((ntr, D)).astype(np.float32), rng.integers(0, K, ntr).astype(np.int32),
                         rng.standard_normal((nte, D)).astype(np.float32), rng.integers(0, K, nte).astype(np.int32))
        ms = fg.time_op('sample_stats', reps=a.reps)
    print(json.dumps(dict(op='sample_stats', precision=a.precision, folds=a.folds, D=D, n_test=nte, ms=round(ms, 4), gpu=gpu_info())))


if __name__ == '__main__':
    main()
