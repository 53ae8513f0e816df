"""CPU suite, part 5: bench.py's reference arm runs without a GPU and prints one JSON line with the contract's keys;
its arguments are checked; (GPU) --dump-outputs writes the same bounded arrays on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_bench_rejects_arguments_it_cannot_honour(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                 ["--workload", "dp", "--dump-outputs", str(tmp_path / "d")]):
        r = _bench(*args)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-2000:])
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_are_bounded_and_identical_from_run_to_run(tmp_path):
    """Two builds are compared through --dump-outputs, so with the same arguments the dump must not change from run to run;
    it holds float32/float64 arrays of at most 64 MB, from exactly --steps timed epochs."""
    runs = []
    for name in ("a", "b"):
        d = tmp_path / name
        r = _bench("--folds", "2", "--steps", "2", "--warmup", "1", "--no-cpu", "--no-modes", "--dump-outputs", str(d), timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2
        files = sorted(os.listdir(d))
        assert files == ["disc_params.npy", "epoch_stats.npy", "gen_params.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        arrays = {f: np.load(d / f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in arrays.values())
        assert arrays["epoch_stats.npy"].shape == (2, 5) and arrays["disc_params.npy"].shape[0] == 2
        runs.append(arrays)
    for f in runs[0]:
        np.testing.assert_array_equal(runs[0][f], runs[1][f])


def test_reference_arm_prints_the_contract_line():
    r = _bench("--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-pairs", "2", "--modality", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "gan_train_step_pairs_per_sec" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "workload" in line["config"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_algorithmic_work_matches_the_survey_table():
    sys.path.insert(0, ROOT)
    import bench
    for D, gf, mb in ((400, 1.456, 46.7), (1200, 2.336, 80.8), (3632, 5.012, 184.4), (12032, 14.25, 542.5)):   # SURVEY.md 8(d)
        flops, nbytes, N_D, N_G = bench.algo_work(D, 50)
        assert abs(flops / 1e9 - gf) < 0.01 * gf and abs(nbytes / 1e6 - mb) < 0.01 * mb
        assert N_D == 1000 * D + 753756 and N_G == 501 * D + 302000
