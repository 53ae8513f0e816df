#!/usr/bin/env python
"""bench.py -- GAN train step-pairs/s (one D step + one G step, mr_gan.py:204-213) on 1..8 B200.

Workload (BASELINE.json configs[2] slice, compact MREO shape): a group of `--folds` independent table-1
fold-trainings per GPU (force+temperature modality, D=1200, N_train=6000, N_test=1200, B=50), synthetic data,
random-init weights.  One bench "step" = ONE EPOCH of the group = 120 D+G step-pairs per fold x folds, launched as
one CUDA graph (plus the batch-wise test pass of mr_gan.py:219-223).  Folds shard over GPUs with no collective
(weak scaling).

  value     : step-pairs/s, device time (CUDA events on the launching stream), fold data and the epoch's index arrays
              already resident in HBM.
  e2e       : the same metric through the public host API (dataset upload + device-side fold preparation + train_epoch
              with HOST numpy index arrays + statistics read-back + final eval), wall clock, H2D / D2H inside.
  roofline  : the kernel with the largest share of the step (dW of D layer 1 with the Adam update fused in), live;
  rooflines : the same arithmetic for every kernel class (forward, dX, dW+Adam), worst first -- the first entry is the
              LIMITING class; step_roofline is the whole step against the algorithmic bytes of SURVEY.md 8(d).
  modes     : the other precision modes on the same workload (short runs), so the fp32 parity mode is on record too.
  dp        : (N > 1 only) BASELINE config 5 measured in the same launch: ONE fold at a large global batch split over
              the N ranks (NCCL all-reduces over NVLink), with its parity against the single-GPU step.
  --impl reference : the restated CPU baseline (oracle/torch_twin.py, torch CPU fp32): one fold per host core, all
              cores busy -- the way a CPU user would run the sweep.  Keras 2.0.9 / Theano 0.9 cannot be installed here
              (SURVEY.md 8c).
  --workload table1 : the whole table-1 sweep (294 fold-trainings, 7 widths) through the drop-in's scheduler, wall clock.
  --dump-outputs DIR : after the timed steps, what the last of them computed (see dump_outputs), so that two builds can be
              compared output for output; the inputs depend only on the arguments.
"""
import argparse
import atexit
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "gan_train_step_pairs_per_sec"
UNIT = "step-pairs/s"
DTYPE = {"fp32": "f32", "tf32": "tf32", "f16": "f16"}      # arithmetic type of the GEMM operands (accumulation is f32)


def algo_work(D, B=50):
    """SURVEY.md 8(d) / BASELINE.md 3: algorithmic FLOPs and bytes per D+G step-pair."""
    P_D = 1000 * D + 751500
    P_G = 500 * D + 300000
    N_D = 1000 * D + 753756
    N_G = 501 * D + 302000
    flops = 2 * B * (9 * P_D + P_G - 3000 * D) + 2 * B * (3 * P_G + 3 * (P_D - 1500) - 50000)
    nbytes = 28 * N_D + 28 * N_G + 4 * (3 * B * D + 2 * B * 100)
    return flops, nbytes, N_D, N_G


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (read-only queries, sampled every period_ms)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_ms=200):
        self.gpu, self.period = gpu_index, period_ms
        self.rows = []
        self.proc = None
        self.reader = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", str(self.period), "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        atexit.register(self._end)      # `nvidia-smi -lms` loops until killed: it must not outlive a run that fails
        self.reader = threading.Thread(target=self._read, daemon=True)
        self.reader.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def _end(self):
        if self.proc.poll() is None:
            self.proc.terminate()
        self.proc.wait()
        self.reader.join(timeout=5)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self._end()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        busy = [s for s in sm if s > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_jobs(D_modality, n_folds, seed):
    """Index-only folds of one synthetic MREO-shape dataset (table 1 reuses X for every labeled % and fold)."""
    from sklearn.model_selection import StratifiedKFold
    from mr_gan_b200 import foldprep, synthetic
    X, y = synthetic.synthetic_dataset(D_modality, seed=seed, dtype=np.float32)
    percents = [100, 50, 16, 8, 4, 2, 1]
    folds = []
    k = 0
    while len(folds) < n_folds:
        skf = StratifiedKFold(n_splits=6, shuffle=True, random_state=seed + k)
        for tr, te in skf.split(X, y):
            if len(folds) < n_folds:
                rng = np.random.default_rng([seed, len(folds)])
                folds.append((foldprep.prepare_fold_indices(y, tr, te, percents[k % len(percents)], None, rng), rng))
        k += 1
    return X, y.astype(np.int32), folds


DUMP_PARAM_VALUES = 1 << 23     # trained parameter values --dump-outputs writes (32 MB of float32), over all folds and both nets


def dump_outputs(path, fg, stats):
    """What a train_epoch caller receives from the last timed step, as float32 .npy files: epoch_stats [folds, 5] (loss_lab,
    loss_unl, train_err, loss_gen, test_err, as returned), and disc_params / gen_params [folds, k]: every fold's trained
    weights at k flat positions (reference weight order) drawn once from a fixed seed -- one fold's weights alone are 11 MB at D=1200."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "epoch_stats.npy"), np.asarray(stats, dtype=np.float32))
    for net, name in ((0, "disc_params"), (1, "gen_params")):
        n = fg.num_params(0, net)                   # every fold of the group has the same width
        pick = np.sort(np.random.default_rng(net).choice(n, min(n, DUMP_PARAM_VALUES // (2 * fg.n_folds)), replace=False))
        rows = [np.concatenate([p.ravel() for p in fg.get_params(i, net)])[pick] for i in range(fg.n_folds)]
        np.save(os.path.join(path, name + ".npy"), np.stack(rows).astype(np.float32))


# ------------------------------------------------------------------ CPU arm (the oracle's torch twin; test infrastructure
# used here only as the measured CPU baseline, never on the product path)
def cpu_pairs_per_sec(D, B, n_pairs, warm=3, threads=None):
    """Restated CPU baseline: torch-CPU fp32 twin, Python loop, two calls per iteration, host noise (mr_gan.py:204-213)."""
    import torch
    from oracle import gan_oracle as O, torch_twin as T
    # torchrun exports OMP_NUM_THREADS=1: use every host thread unless a thread count is asked for
    torch.set_num_threads(threads or max(1, os.cpu_count() or 1))
    rng = np.random.default_rng(0)
    m = T.TorchGan(O.init_disc_params(D, rng), O.init_gen_params(D, rng), dtype=torch.float32)
    X = rng.standard_normal((6000, D)).astype(np.float32)
    y = rng.integers(0, 6, 6000)

    def pair(t):
        sl = slice((t % 100) * B, (t % 100 + 1) * B)
        noise = np.random.normal(0, 1, size=[B, 100]).astype(np.float32)
        m.disc_step(X[sl], y[sl], X[sl], noise)
        noise = np.random.normal(0, 1, size=[B, 100]).astype(np.float32)
        m.gen_step(X[sl], noise)
    for t in range(warm):
        pair(t)
    t0 = time.perf_counter()
    for t in range(n_pairs):
        pair(t)
    dt = time.perf_counter() - t0
    return n_pairs / dt, torch.get_num_threads()


def _core_worker(args):
    D, B, warm_pairs, n_pairs, barrier = args
    os.environ["OMP_NUM_THREADS"] = "1"
    import torch
    from oracle import gan_oracle as O, torch_twin as T
    torch.set_num_threads(1)
    rng = np.random.default_rng(os.getpid())
    m = T.TorchGan(O.init_disc_params(D, rng), O.init_gen_params(D, rng), dtype=torch.float32)
    X = rng.standard_normal((6000, D)).astype(np.float32)
    y = rng.integers(0, 6, 6000)

    def pair(t):
        sl = slice((t % 100) * B, (t % 100 + 1) * B)
        m.disc_step(X[sl], y[sl], X[sl], np.random.normal(0, 1, size=[B, 100]).astype(np.float32))
        m.gen_step(X[sl], np.random.normal(0, 1, size=[B, 100]).astype(np.float32))
    for t in range(max(1, warm_pairs)):
        pair(t)
    barrier.wait()
    t0 = time.perf_counter()
    for t in range(n_pairs):
        pair(t)
    return n_pairs, time.perf_counter() - t0


def cpu_fold_per_core(D, B, warm_pairs, n_pairs, cores=None):
    """One independent fold-training per host core (torch threads = 1 each), all cores busy at once: how the reference's
    table sweeps would be spread over a CPU box.  Returns (aggregate step-pairs/s, cores, slowest worker's seconds)."""
    cores = cores or max(1, os.cpu_count() or 1)
    ctx = mp.get_context("spawn")
    with ctx.Manager() as mgr:
        barrier = mgr.Barrier(cores)
        with ctx.Pool(cores) as pool:
            res = pool.map(_core_worker, [(D, B, warm_pairs, n_pairs, barrier)] * cores)
    slowest = max(s for _, s in res)
    return sum(n for n, _ in res) / slowest, cores, slowest


def sweep_workload(G, D, ntr, nte, B):
    """config.workload of the sweep bench: ONE string for both arms (the reference arm times a bounded sample of it)."""
    return ("mr_gan.py table-1 fold group: %d folds/GPU, force+temperature D=%d, N_train=%d, N_test=%d, B=%d; "
            "1 step = 1 epoch = %d D+G step-pairs per fold + test pass" % (G, D, ntr, nte, B, ntr // B))


def run_reference(args, rank):
    if rank != 0:
        return 0
    D, B = args.width, 50
    t0 = time.perf_counter()
    v, cores, secs = cpu_fold_per_core(D, B, max(1, args.warmup) * args.ref_pairs, args.steps * args.ref_pairs)
    v_one, threads = cpu_pairs_per_sec(D, B, max(4, args.ref_pairs), warm=2)
    sample = ("one fold per host core: %d cores x %d steps x %d step-pairs (D=%d, B=%d), torch-CPU fp32 twin of the oracle, "
              "1 thread per fold" % (cores, args.steps, args.ref_pairs, D, B))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "wall_ms": 1e3 * (time.perf_counter() - t0),
            # the b200 arm's workload (table-1 split of 7200 rows: 6000 train / 1200 test); each step here is a bounded sample
            # of it -- args.ref_pairs step pairs of one fold per host core -- described in cpu_baseline.sample
            "config": {"workload": sweep_workload(args.folds, D, 6000, 1200, B), "folds_per_gpu": args.folds, "D": D, "batch": B,
                       "precision": "fp32 (torch CPU)", "parallelism": "one fold per host core, %d cores" % cores},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "host_cpus": os.cpu_count(),
                             "value_one_fold_all_threads": v_one, "threads_one_fold": threads},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------ data-parallel large-batch measurement (config 5)
def measure_dp(args, precision, rank, world, local, barrier, min_seconds=1.5, parity=True):
    """ONE fold at a large global batch, batch rows split over the ranks; BN / feature-matching statistics and the flat
    gradient all-reduced with NCCL over NVLink (strong scaling: the global batch is fixed).  Returns the record dict."""
    import torch
    import torch.distributed as dist
    from mr_gan_b200.engine import FoldGroup
    from mr_gan_b200.model import init_disc, init_gen
    D, Bg, nb = args.dp_width, args.dp_batch, 2
    Bl = Bg // world
    rng = np.random.default_rng(0)                      # identical on every rank: weights and the GLOBAL batches
    pD, pG = init_disc(D, rng), init_gen(D, rng)
    Xg = rng.standard_normal((nb * Bg, D), dtype=np.float32)
    yg = (np.arange(nb * Bg) % 6).astype(np.int32)
    rows = np.concatenate([np.arange(t * Bg + rank * Bl, t * Bg + (rank + 1) * Bl) for t in range(nb)])
    fg = FoldGroup([(D, nb * Bl, 600, 4242)], precision=precision, batch=Bl, device=local, eval_each_epoch=False)
    if world > 1:
        uid = [FoldGroup.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)

        def allgather(b):                               # CUDA IPC handles of every rank's arena: fused peer-memory exchange
            out = [None] * world
            dist.all_gather_object(out, b)
            return out
        fg.dp_init(rank, world, uid[0], allgather=None if os.environ.get("MRGAN_DP_FUSED") == "0" else allgather)
    fg.set_params(0, 1, pG)
    fg.set_params(0, 0, pD)
    fg.load_fold(0, Xg[rows], yg[rows], Xg[:600], yg[:600])
    idx = np.arange(nb * Bl, dtype=np.int32)[None, :]
    first = fg.train_epoch(idx, idx, idx)[0]            # epoch 0 from the initial weights: the parity sample
    for w in range(2):
        fg.train_epoch(idx, idx, idx)
    sampler = ClockSampler(local, period_ms=100)
    sampler.start()
    barrier()
    l0 = fg.kernel_launches
    t0 = time.perf_counter()
    dev_ms, K = 0.0, 0
    while K < 3 or time.perf_counter() - t0 < min_seconds:
        st = fg.train_epoch(idx, idx, idx)
        dev_ms += fg.last_device_ms
        K += 1
        if world > 1:                                   # every rank must stop after the same epoch
            flag = torch.tensor([K >= 3 and time.perf_counter() - t0 >= min_seconds], dtype=torch.int32, device="cuda")
            dist.broadcast(flag, src=0)
            if int(flag.item()):
                break
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    launches = fg.kernel_launches - l0
    fg.close()
    t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = (float(x) for x in t.tolist())
    pairs = K * nb
    flops, nbytes, N_D, N_G = algo_work(D, Bg)
    hbm, tf, how = peaks()
    value = pairs / (dev_ms * 1e-3)
    ach = flops * value / 1e12
    rec = {"value": value, "unit": UNIT, "ms_per_pair": dev_ms / pairs, "epochs_timed": K, "pairs_per_epoch": nb,
           "workload": "mr_gan.py table-5 fold at large batch, data-parallel: D=%d (1 s contact mic), global batch %d (%d per GPU)"
                       % (D, Bg, Bl),
           "parallelism": "dp%d: %s of the flat gradients (%.0f MB D + %.0f MB G per pair); NCCL all-reduce of the BN / "
                          "feature-matching statistics; epoch captured as one CUDA graph"
                          % (world, "NCCL all-reduce + full Adam" if os.environ.get("MRGAN_DP_FUSED") == "0" or world == 1 else
                             "fused peer-memory reduce-scatter + sharded Adam + all-gather (k_dp_exchange)", 4e-6 * N_D, 4e-6 * N_G),
           "precision": precision, "scaling": "strong", "e2e_value": pairs / (wall_ms * 1e-3), "gpu_launches": int(launches),
           "achieved_tflops": ach, "tensor_frac_of_bf16_peak": ach / (tf * world), "peak_source": how, "clocks": clocks,
           "last_loss_lab": float(st[0, 0]), "last_loss_gen": float(st[0, 3])}
    if parity and world > 1:
        # the same global batches through ONE GPU's large-batch step, from the same weights: epoch 0 must agree
        ref = None
        if rank == 0:
            with FoldGroup([(D, nb * Bg, 600, 4242)], precision=precision, batch=Bg, device=local, eval_each_epoch=False) as f1:
                f1.set_params(0, 1, pG)
                f1.set_params(0, 0, pD)
                f1.load_fold(0, Xg, yg, Xg[:600], yg[:600])
                i1 = np.arange(nb * Bg, dtype=np.int32)[None, :]
                ref = f1.train_epoch(i1, i1, i1)[0]
            rel = np.abs(first[[0, 1, 3]] - ref[[0, 1, 3]]) / np.abs(ref[[0, 1, 3]])
            rec["parity_vs_single_gpu"] = {"max_rel_err_losses": float(rel.max()), "train_err_abs_diff": float(abs(first[2] - ref[2])),
                                           "dp": [float(x) for x in first[:4]], "single_gpu": [float(x) for x in ref[:4]]}
        barrier()
    return rec


def run_dp(args, rank, world, local, barrier):
    import torch.distributed as dist
    rec = measure_dp(args, args.precision, rank, world, local, barrier, min_seconds=max(1.5, 0.05 * args.steps))
    hbm, tf, how = peaks()
    line = {"metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": rec["epochs_timed"], "warmup": 3,
            "ms_per_step": rec["ms_per_pair"] * rec["pairs_per_epoch"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": rec["workload"], "parallelism": rec["parallelism"], "precision": args.precision},
            "e2e": {"value": rec["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": int(3 * 4 * rec["pairs_per_epoch"] * args.dp_batch // world),
                    "d2h_bytes_per_step": 32},
            "gpu_launches": rec["gpu_launches"],
            "roofline": {"kernel": "whole step pair (tcgen05 GEMMs dominate at this batch)", "bound": "tensor",
                         "achieved": rec["achieved_tflops"], "peak": tf * world, "unit": "TFLOP/s",
                         "frac": rec["tensor_frac_of_bf16_peak"], "traffic": None, "peak_source": how,
                         "note": "denominator = measured bf16 cuBLAS throughput; tf32 operands run at half that rate"},
            "clocks": rec["clocks"], "dp": rec}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------ the whole table-1 sweep through the drop-in scheduler
def run_table1(args, rank, world, local, barrier):
    import torch.distributed as dist
    from mr_gan_b200 import mr_gan as mg, sweep
    t0 = time.perf_counter()
    seed = 0
    percents = [1, 2, 4, 8, 16, 50, 100]
    jobs = []
    for modality in range(len(mg.MODALITIES)):
        X, y = mg.dataset(modalities=modality, seed=seed, synthetic_data=True)
        jobs += [j for p in percents for j in mg._kfold_jobs(X, y, seed + p, percentlabeled=p)]
    for i, j in enumerate(jobs):
        j['job_id'] = i
    t_data = time.perf_counter() - t0
    errors = sweep.run_sharded(jobs, lambda js, dev: mg.train_gan_folds(js, epochs=args.epochs, seed=seed, precision=args.precision, device=dev),
                               group_size=args.group, key=mg.job_rows, cost=mg.job_cost, init_dist=False)
    barrier()
    wall = time.perf_counter() - t0
    pairs = sum((mg.job_rows(j)[0] // 50) * args.epochs for j in jobs)
    line = {"metric": "table1_sweep_wall_seconds", "value": wall, "unit": "s", "n_gpus": world, "steps": 1, "warmup": 0,
            "ms_per_step": 1e3 * wall, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": "mr_gan.py --tables 1: %d fold-trainings (7 modalities x 7 labeled fractions x 6 folds), %d epochs, "
                                   "widths 400..3632, through the drop-in scheduler (data synthesis %.1f s included)"
                                   % (len(jobs), args.epochs, t_data), "group": args.group, "precision": args.precision},
            "step_pairs_total": pairs, "step_pairs_per_sec_wall": pairs / wall, "mean_test_error": float(np.mean(errors))}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--folds", type=int, default=74, help="fold-trainings grouped per GPU (table 1 has 294 = 4 x 73.5; 74 = 148/2 keeps every kernel at whole waves)")
    ap.add_argument("--modality", type=int, default=2, help="2 = force+temperature (D=1200)")
    ap.add_argument("--precision", default=os.environ.get("MRGAN_PRECISION", "f16"), choices=["fp32", "tf32", "f16"])
    ap.add_argument("--ref-pairs", type=int, default=6, help="--impl reference: step-pairs per fold and step (bounded CPU sample)")
    ap.add_argument("--cpu-pairs", type=int, default=30)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-modes", action="store_true", help="skip the short runs of the other precision modes")
    ap.add_argument("--no-dp", action="store_true", help="N > 1: skip the data-parallel sub-record")
    ap.add_argument("--workload", default="sweep", choices=["sweep", "dp", "table1"],
                    help="sweep: fold-sharded table-1 group (headline); dp: ONE fold at large batch, data-parallel (config 5); "
                         "table1: the whole table-1 sweep, wall clock")
    ap.add_argument("--dp-batch", type=int, default=8192, help="global batch of the dp workload")
    ap.add_argument("--dp-width", type=int, default=12032, help="input width of the dp workload (1 s contact mic, table 5)")
    ap.add_argument("--epochs", type=int, default=100, help="table1 workload: epochs per fold")
    ap.add_argument("--group", type=int, default=84, help="table1 workload: largest number of folds per handle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="sweep workload: write what the last timed step computed to DIR/*.npy "
                                                          "(rank 0's folds; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "sweep"):
        ap.error("--dump-outputs applies to the sweep workload of the b200 arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from mr_gan_b200 import synthetic
    args.width = synthetic.feature_width(args.modality)
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from mr_gan_b200 import foldprep
    from mr_gan_b200.engine import FoldGroup
    from mr_gan_b200.model import fold_key, init_disc, init_gen

    if args.workload == "dp":
        return run_dp(args, rank, world, local, barrier)
    if args.workload == "table1":
        return run_table1(args, rank, world, local, barrier)

    D, B, G = args.width, 50, args.folds
    W, K = max(args.warmup, 3), args.steps
    X, y, folds = make_jobs(args.modality, G, seed=1000 * rank)
    ntr, nte = len(folds[0][0].train_rows), len(folds[0][0].test_rows)
    nb = ntr // B

    def draw():
        per = [foldprep.epoch_indices(rng, ntr, f.lab_rows, f.unl_rows) for f, rng in folds]
        return [np.stack([p[s] for p in per]) for s in range(3)]

    def open_group(precision):
        fg = FoldGroup([(D, ntr, nte, fold_key(rank, i)) for i in range(G)], precision=precision, device=local)
        for i, (f, rng) in enumerate(folds):
            r2 = np.random.default_rng([7, rank, i])
            fg.set_params(i, 1, init_gen(D, r2))
            fg.set_params(i, 0, init_disc(D, r2))
        return fg

    def load_all(fg):        # dataset upload (once) + device-side fold preparation of every fold (scaler, gather)
        fg.load_dataset(0, X, y)
        for i, (f, rng) in enumerate(folds):
            fg.prepare_fold(i, 0, f.train_rows, f.test_rows)

    fg = open_group(args.precision)
    load_all(fg)
    pre = [draw() for _ in range(W + K)]

    sampler = ClockSampler(local)
    for w in range(W):
        fg.train_epoch(*pre[w])
    sampler.start()
    # ---- region 1: device-timed, inputs resident -------------------------------------------
    barrier()
    l0 = fg.kernel_launches
    t0 = time.perf_counter()
    dev_ms = 0.0
    for k in range(K):
        st = fg.train_epoch(*pre[W + k])
        dev_ms += fg.last_device_ms
    barrier()
    wall1 = time.perf_counter() - t0
    launches = fg.kernel_launches - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fg, st)
    # ---- region 2: end to end through the host API -----------------------------------------
    barrier()
    t0 = time.perf_counter()
    load_all(fg)                                          # H2D of the dataset + per-fold index arrays, fold prep on the device
    for i, (f, rng) in enumerate(folds):
        fg.set_epoch_rows(i, f.lab_rows, f.unl_rows)      # labeled rows of every fold: the epoch permutations are drawn on the device
    t_load = time.perf_counter() - t0
    for k in range(K):
        fg.train_epoch_seeded(k, wait=False)              # H2D per epoch: one epoch number (mr_gan.py:189-202 run on the device)
        st = fg.epoch_result()                            # D2H of the epoch statistics
    t_train = time.perf_counter() - t0 - t_load
    errs = [fg.eval(i) for i in range(G)]
    barrier()
    wall2 = time.perf_counter() - t0
    t_eval = wall2 - t_train - t_load
    clocks = sampler.stop()

    t = torch.tensor([dev_ms, wall1 * 1e3, wall2 * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall1_ms, wall2_ms = (float(x) for x in t.tolist())
    pairs = K * nb * G * world
    value = pairs / (dev_ms * 1e-3)
    e2e = pairs / (wall2_ms * 1e-3)

    # ---- live roofline probes, one per kernel class (CUDA events on the launching stream; they mutate the state, so
    #      they run after the measured regions) ----
    flops, nbytes, N_D, N_G = algo_work(D, B)
    hbm, tf, how = peaks()
    tensor = args.precision != "fp32"
    wbytes = 2 if args.precision == "f16" else 4            # bytes per weight the forward / dX passes read
    probe = {k: fg.time_op(k, reps=10) for k in ("adam_d", "dw1", "fwd1", "dx1", "adam_g")}
    step_ms = {k: fg.time_op(k, reps=3) for k in ("disc_step", "gen_step")}
    n1 = (D + 1) * 1000                                       # parameters of D layer 1 (augmented: bias row included)
    adam_bytes = 24.0 + (2.0 if args.precision == "f16" else 0.0)   # W, m, v read + written (+ the fp16 operand copy written)

    def hbm_entry(name, kernel, ms, per_param, n_par, note):
        ach = per_param * n_par * G / (ms * 1e-3) / 1e9
        return {"class": name, "kernel": kernel, "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                "launch_ms": ms, "algorithmic_bytes_per_launch": per_param * n_par * G, "bytes_per_parameter": per_param,
                "peak_source": how, "note": note}

    if tensor:
        classes = [
            hbm_entry("dW + fused Adam", "k_dw_adam_tc, D layer 1, all folds", probe["dw1"], adam_bytes, n1,
                      "W, m, v streamed once each way; the gradient never leaves the SM"),
            hbm_entry("forward", "k_gemm_tc<forward>, D layer 1, all folds", probe["fwd1"], wbytes, n1,
                      "weights read once; the 150-row activation tile is L2-resident and not counted"),
            hbm_entry("dX", "k_gemm_tc<dX>, dFake = dZ1 W1^T, all folds", probe["dx1"], wbytes, D * 1000,
                      "weights read once; 50 gradient rows L2-resident"),
        ]
    else:
        classes = [
            hbm_entry("flat Adam", "k_adam, discriminator, all folds", probe["adam_d"], 24.0, N_D,
                      "W, m, v read + written; the gradient read (4 B) is not algorithmic"),
            {"class": "forward", "kernel": "k_gemm_simt, D layer 1, all folds", "bound": "fp32 FFMA", "launch_ms": probe["fwd1"],
             "achieved": 2.0 * 3 * B * n1 * G / (probe["fwd1"] * 1e-3) / 1e12, "unit": "TFLOP/s", "peak": None, "frac": None},
        ]
    rooflines = sorted([c for c in classes if c.get("frac") is not None], key=lambda c: c["frac"])
    dominant = dict(classes[0])                               # largest share of the step (profiles/: launch list)
    # dram__bytes_read + dram__bytes_write of that kernel from `ncu --set full`, valid only for the library it was captured
    # on (keyed by the source hash): a stale constant is worse than null
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        from mr_gan_b200 import build as _b
        tj = json.load(open(tpath)).get("dw1/%s" % args.precision, {})
        if tj.get("folds") == G and tj.get("D") == D and tj.get("source_hash") == _b.source_hash():
            traffic = tj["bytes"]
    dominant["traffic"] = traffic
    dominant["limiting_class"] = rooflines[0]["class"] if rooflines else None
    step_gbs = nbytes * value / world / 1e9
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": sweep_workload(G, D, ntr, nte, B),
                       "folds_per_gpu": G, "D": D, "batch": B, "precision": args.precision,
                       "l2": "state of the group (%.0f MB) exceeds L2; no flush needed" % (12e-6 * (N_D + N_G) * G),
                       "parallelism": "fold-sharded x%d, no collective" % world},
            "e2e": {"value": e2e, "unit": UNIT,
                    "h2d_bytes_per_step": int(4 + (X.nbytes + y.nbytes + 4 * (ntr + nte) * G + sum(4 * len(f.lab_rows) for f, _ in folds)) / K),
                    "d2h_bytes_per_step": int(G * 8 * 4), "wall_ms": wall2_ms,
                    "breakdown_ms": {"load_and_prepare_folds": 1e3 * t_load, "epochs": 1e3 * t_train, "final_eval": 1e3 * t_eval},
                    "note": "includes the dataset upload, device-side fold preparation and labeled-row upload once (amortised over the "
                            "steps), per epoch an epoch number up and the statistics down (permutations drawn on the device), final eval"},
            "gpu_launches": int(launches), "wall_ms_region1": wall1_ms,
            "fold_trainings_per_hour": value / (100 * nb) * 3600.0,
            "roofline": dominant, "rooflines": rooflines,
            "step_roofline": {"bound": "hbm", "achieved": step_gbs, "peak": hbm, "unit": "GB/s", "frac": step_gbs / hbm,
                              "algorithmic_bytes_per_pair": nbytes, "algorithmic_flops_per_pair": flops,
                              "achieved_tflops": flops * value / world / 1e12},
            "kernel_ms": probe, "step_ms": step_ms, "clocks": clocks,
            "sanity": {"final_test_err_mean": float(np.mean(errs)), "last_loss_lab": float(st[:, 0].mean())}}
    fg.close()

    # ---- the other precision modes on the same workload (short: 1 warm-up epoch beyond the graph build, 2 timed) ----
    if not args.no_modes:
        modes = {args.precision: {"value": value, "steps": K}}
        for prec in ("f16", "tf32", "fp32"):
            if prec == args.precision:
                continue
            f2 = open_group(prec)
            load_all(f2)
            f2.train_epoch(*pre[0])
            f2.train_epoch(*pre[1])
            barrier()
            ms = 0.0
            for k in range(2):
                f2.train_epoch(*pre[2 + k])
                ms += f2.last_device_ms
            tt = torch.tensor([ms], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            v2 = 2 * nb * G * world / (float(tt.item()) * 1e-3)
            modes[prec] = {"value": v2, "steps": 2, "step_roofline_frac": nbytes * v2 / world / 1e9 / hbm}
            f2.close()
        line["modes"] = modes

    if rank == 0 and world == 1 and not args.no_cpu:
        v, threads = cpu_pairs_per_sec(D, B, args.cpu_pairs)
        vc, cores, _ = cpu_fold_per_core(D, B, 2, max(4, args.cpu_pairs // 3))
        line["cpu_baseline"] = {"value": vc, "unit": UNIT, "cores": cores, "kind": "port", "host_cpus": os.cpu_count(),
                                "value_one_fold_all_threads": v, "threads_one_fold": threads,
                                "sample": "one fold per host core, %d D+G step-pairs each (D=%d, B=%d), torch-CPU fp32 twin of the "
                                          "oracle, 1 thread per fold (restated baseline, not Keras 2.0.9/Theano 0.9); "
                                          "value_one_fold_all_threads = %d step-pairs of ONE fold on all threads"
                                          % (max(4, args.cpu_pairs // 3), D, B, args.cpu_pairs)}
    if world > 1 and not args.no_dp:
        dp_prec = args.precision
        line["dp"] = measure_dp(args, dp_prec, rank, world, local, barrier)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
