"""CPU suite, part 2: host logic (fold prep, permutations, synthetic shapes, scheduler, CLI) and
the C-ABI library surface (loads, exports every declared symbol, fails loudly without a GPU)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from mr_gan_b200 import _lib, foldprep, model, mr_gan as mg, mr_nn as mn, sweep, synthetic
from oracle import fold_loop, philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fold_prep_matches_oracle_restatement():
    X, y = synthetic.synthetic_dataset(1, forcetempTime=0.2, pokes=4, seed=3)      # [288, 20]
    tr, te = np.arange(0, 288, 1)[::2], np.arange(1, 288, 2)
    for pl, pu in ((0.2, None), (0.1, 0.1)):
        f = foldprep.prepare_fold(None, None, pl, pu, [X[tr], X[te], y[tr], y[te]], np.random.default_rng(9))
        o = fold_loop.prep_fold(X[tr], X[te], y[tr], y[te], pl, pu, np.random.default_rng(9))
        np.testing.assert_allclose(f.x_train, o[0], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(f.x_test, o[1], rtol=1e-5, atol=1e-6)
        np.testing.assert_array_equal(f.y_train, o[2])
        np.testing.assert_array_equal(f.lab_rows, o[4])
        if pu is None:
            assert f.unl_rows is None
        else:
            np.testing.assert_array_equal(f.unl_rows, o[5])
        # labeled subset: first 10*percent rows per class, class-major (mr_gan.py:102-103)
        n = int(10 * pl)
        assert list(f.y_train[f.lab_rows]) == [j for j in range(6) for _ in range(n)]
        assert abs(f.x_train.mean()) < 1e-5 and abs(f.x_train.std() - 1) < 1e-3


def test_epoch_indices_match_oracle_and_reference_structure():
    lab_rows = np.array([3, 5, 7, 11, 13])
    a = foldprep.epoch_indices(np.random.default_rng(1), 23, lab_rows)
    b = fold_loop.epoch_indices(np.random.default_rng(1), 23, lab_rows)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v)
        assert u.dtype == np.int32 and u.shape == (23,)
    # mr_gan.py:189: 4 full permutations of the 5 labeled rows then a permutation of the first 3
    for k in range(4):
        assert sorted(a[0][5 * k:5 * k + 5]) == sorted(lab_rows)
    assert sorted(a[0][20:]) == sorted(lab_rows[:3])
    assert sorted(a[1]) == list(range(23)) and sorted(a[2]) == list(range(23)) and not (a[1] == a[2]).all()
    # table-6 path (mr_gan.py:197-200): streams drawn from the unlabeled subset only
    unl = np.array([0, 1, 2, 3, 4, 5, 6, 7])
    c = foldprep.epoch_indices(np.random.default_rng(2), 23, lab_rows, unl)
    assert set(c[1]) <= set(unl) and set(c[2]) <= set(unl)


def test_synthetic_shapes_follow_reference_feature_layout():
    assert [synthetic.feature_width(m) for m in range(7)] == [800, 400, 1200, 2432, 2832, 3632, 3232]
    assert [synthetic.feature_width(3, contactmicTime=c) for c in (1, 0.7, 0.5, 0.3, 0.2, 0.1, 0.05)] == \
        [12032, 8448, 6016, 3712, 2432, 1280, 640]
    assert [synthetic.feature_width(2, forcetempTime=t) for t in (4, 3, 2, 1, 0.5, 0.2, 0.1)] == \
        [1200, 900, 600, 300, 150, 60, 30]
    X, y = synthetic.synthetic_dataset(1, pokes=5, seed=0)
    assert X.shape == (360, 400) and list(np.bincount(y)) == [60] * 6
    X2, _ = synthetic.synthetic_dataset(1, pokes=5, seed=0)
    np.testing.assert_array_equal(X, X2)
    objs = synthetic.synthetic_dataset(1, pokes=5, seed=0, leaveObjectOut=True)
    assert len(objs) == 72 and all(o['x'].shape == (5, 400) for o in objs.values())


def test_model_shapes_and_parameter_counts():
    for D in (10, 400, 1200, 3632):
        assert sum(int(np.prod(s)) for s in model.disc_shapes(D)) == 1000 * D + 753756      # SURVEY.md 8
        assert sum(int(np.prod(s)) for s in model.gen_shapes(D)) == 501 * D + 302000
    p = model.init_gen(30, np.random.default_rng(0))
    assert (p[2] == 1).all() and (p[3] == 0).all() and (p[1] == 0).all()
    w = model.init_disc(30, np.random.default_rng(0))[0]
    assert np.abs(w).max() <= np.sqrt(6.0 / (30 + 1000)) and w.dtype == np.float32
    lo, hi = philox.fold_key(77, 5)
    assert model.fold_key(77, 5) == (hi << 32) | lo


def test_sweep_grouping_and_assignment():
    jobs = [dict(n=6000, D=d) for d in (800, 800, 400, 1200, 1200, 1200, 1200)] + [dict(n=7100, D=800)]
    groups = sweep.make_groups(jobs, 3, key=lambda j: j['n'])
    assert groups == [[0, 1, 2], [3, 4, 5], [6], [7]]
    owner = sweep.assign(groups, 2, [sum(jobs[i]['D'] for i in g) for g in groups])
    loads = [sum(sum(jobs[i]['D'] for i in g) for g, o in zip(groups, owner) if o == r) for r in (0, 1)]
    assert max(loads) <= 4000 and sorted(set(owner)) == [0, 1]
    res = sweep.run_sharded(jobs, lambda js, dev: [j['D'] * 2 for j in js], group_size=3, key=lambda j: j['n'])
    assert res == [2 * j['D'] for j in jobs]


def test_sweep_plan_deals_folds_by_cost_over_ranks():
    """Table 1 on 8 GPUs: 7 modalities x 42 folds of widths 400..3632 (mr_gan.py:49-62,248-258).  Every fold is trained
    exactly once, groups share (n_train, n_test), and no rank carries more than 1 % above the mean cost -- dealing whole
    one-modality groups left one GPU idle and the widest modality alone on another."""
    widths = [800, 400, 1200, 2432, 2832, 3632, 3232]
    jobs = [dict(D=widths[m], n=6000 if m != 3 else 7100) for m in range(7) for _ in range(42)]
    cost = lambda j: (j['D'] + 703.0) * (j['n'] // 50)
    for world in (1, 2, 4, 8):
        pl = sweep.plan(jobs, world, 42, key=lambda j: j['n'], cost=cost)
        seen = sorted(i for r in pl for g in pl[r] for i in g)
        assert seen == list(range(len(jobs)))
        assert all(len(g) <= 42 and len({jobs[i]['n'] for i in g}) == 1 for r in pl for g in pl[r])
        if world > 1:
            loads = [sum(cost(jobs[i]) for g in pl[r] for i in g) for r in range(world)]
            assert max(loads) <= 1.01 * sum(loads) / world, loads
    one = sweep.plan(jobs, 1, 42, key=lambda j: j['n'], cost=cost)[0]
    assert one == sweep.make_groups(jobs, 42, key=lambda j: j['n'])        # one GPU: the reference's loop order, cut into groups
    # inside a mixed group the concurrent fold chains (contiguous quarters of the group) carry equal cost
    g = sweep.plan(jobs, 8, 42, key=lambda j: j['n'], cost=cost)[0][0]
    nch = sweep.chain_count(len(g))
    q = [sum(cost(jobs[i]) for i in g[len(g) * ch // nch:len(g) * (ch + 1) // nch]) for ch in range(nch)]
    assert nch == 4 and max(q) <= 1.15 * min(q), q


def test_dataset_raises_without_the_pickles_unless_synthetic_is_requested(tmp_path):
    """The reference's dataset() raises IOError on a missing pickle (mr_gan.py:33 open()); so does the drop-in.  Synthetic
    data is opt-in: a wrong --data-dir must not print plausible tables from made-up data."""
    with pytest.raises(IOError):
        mg.dataset(modalities=1, data_dir=str(tmp_path / "nope"))
    X, y = mg.dataset(modalities=1, data_dir=str(tmp_path / "nope"), synthetic_data=True)
    assert X.shape == (7200, 400) and y.shape == (7200,)
    assert sweep.shared_seed(7) == 7 and 0 <= sweep.shared_seed(None) < 2 ** 31


def test_build_is_content_hashed_and_abi_checked():
    from mr_gan_b200 import build as B
    assert not B._stale()                       # the suite built / loaded it already
    h = B.source_hash()
    assert open(B.HASH).read().strip() == h
    lib = _lib.load()
    info = (C.c_int * 4)()
    assert lib.mrgan_abi_info(info) == 0
    assert list(info) == [_lib.ABI_VERSION, C.sizeof(_lib.Config), C.sizeof(_lib.FoldShape), C.sizeof(_lib.EpochStats)]


def test_cli_surface_matches_reference_flags():
    for mod in (mg, mn):
        with pytest.raises(SystemExit):
            mod.main([])                                       # --tables is required (mr_gan.py:240)
    assert mg.MODALITIES[5] == 'Force, Temperature, and Contact Mic'
    jobs = mg._kfold_jobs(*synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=2, seed=0), 0, percentlabeled=1)
    assert len(jobs) == 6 and mg.job_rows(jobs[0]) == (120, 24) and mg.job_width(jobs[0]) == 10
    loo = mg._loo_jobs(synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=2, seed=0, leaveObjectOut=True), percentlabeled=1)
    assert len(loo) == 72 and mg.job_rows(loo[0]) == (142, 2) and mg.job_width(loo[0]) == 10
    assert sorted(np.concatenate([loo[5]['train_idx'], loo[5]['test_idx']])) == list(range(144))
    # index-only fold prep draws from the generator exactly like the host path and picks the same rows
    X, y = synthetic.synthetic_dataset(1, forcetempTime=0.1, pokes=2, seed=0)
    j = jobs[0]
    fi = foldprep.prepare_fold_indices(y, j['train_idx'], j['test_idx'], 0.1, 0.1, np.random.default_rng(5))
    fh = foldprep.prepare_fold(None, None, 0.1, 0.1, [X[j['train_idx']], X[j['test_idx']], y[j['train_idx']], y[j['test_idx']]],
                               np.random.default_rng(5))
    np.testing.assert_array_equal(fi.y_train, fh.y_train)
    np.testing.assert_array_equal(fi.lab_rows, fh.lab_rows)
    np.testing.assert_array_equal(fi.unl_rows, fh.unl_rows)
    np.testing.assert_array_equal(y[fi.train_rows], fh.y_train)


# ------------------------------------------------------------------ C-ABI surface (no compute)
def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "mrgan.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mr(?:gan|nn)_[a-z_]+)\s*\(", src)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 20
    assert sorted(_lib.SYMBOLS) == declared            # the ctypes table and the header agree
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.mrgan_version()
    cfg = _lib.Config()
    assert lib.mrgan_default_config(0, C.byref(cfg)) == 0
    assert (cfg.batch, cfg.n_classes, cfg.noise_dim, cfg.shared_t) == (50, 6, 100, 1)       # mr_gan.py:77-80
    assert np.isclose(cfg.lr, 6e-4) and np.isclose(cfg.beta1, 0.5) and np.isclose(cfg.bn_eps, 2e-5)
    assert lib.mrgan_default_config(1, C.byref(cfg)) == 0
    assert cfg.batch == 20 and np.isclose(cfg.lr, 1e-3) and np.isclose(cfg.beta1, 0.9)      # mr_nn.py:114,117


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mr_gan_b200.engine import FoldGroup, MrganError
    with pytest.raises(MrganError, match="no CPU fallback"):
        FoldGroup([(16, 100, 20, 1)])


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "mr_gan_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn
    code = "import sys; import mr_gan_b200; assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules)"
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)


def test_scheduler_mirrors_the_library_chain_rule(monkeypatch):
    """sweep.chain_count restates how mrgan_create splits a group into concurrent fold chains; order_for_chains balances
    exactly those ranges, so the two must not drift apart: the rule is read back from the C source."""
    import re
    src = open(os.path.join(ROOT, "mr_gan_b200", "csrc", "mrgan_api.cu")).read()
    m = re.search(r"h->nf >= (\d+) \? (\d+) : \(h->nf >= (\d+) \? (\d+) : (\d+)\)", src)
    assert m, "chain rule not found in mrgan_api.cu"
    a, na, b, nb_, nc = map(int, m.groups())
    kmax = int(re.search(r"constexpr int kMaxChains = (\d+);", src).group(1))
    monkeypatch.delenv("MRGAN_CHAINS", raising=False)
    for nf in (1, 2, b - 1, b, a - 1, a, 500):
        want = na if nf >= a else (nb_ if nf >= b else nc)
        assert sweep.chain_count(nf) == max(1, min(want, kmax, nf))
    monkeypatch.setenv("MRGAN_CHAINS", "12")
    assert sweep.chain_count(74) == 12 and sweep.chain_count(5) == 5
    monkeypatch.setenv("MRGAN_CHAINS", "999")
    assert sweep.chain_count(74) == kmax


def test_library_has_one_code_path_per_decision():
    """The library is built one way and measured one way: no build-time variant, no environment switch that selects an
    alternative kernel path, no programmatic-dependent-launch hooks, no opt-in BatchNorm-backward head.  The two variables
    it does read are a scheduling parameter (MRGAN_CHAINS) and a numeric one (MRGAN_LOSS_SCALE)."""
    csrc = os.path.join(ROOT, "mr_gan_b200", "csrc")
    names = sorted(os.listdir(csrc))
    assert "mrgan_api.cu" in names and "kernels_tc.cuh" in names
    for fn in names:
        src = open(os.path.join(csrc, fn)).read()
        for word in ("MRGAN_WITH_TC", "griddepcontrol", "HEAD_BN_BWD"):
            assert word not in src, (fn, word)
        calls = re.findall(r"\bgetenv\s*\(", src)
        read = re.findall(r"\bgetenv\s*\(\s*\"(\w+)\"\s*\)", src)
        assert len(read) == len(calls), (fn, "getenv of a non-literal name")
        assert set(read) <= {"MRGAN_CHAINS", "MRGAN_LOSS_SCALE"}, (fn, read)


def test_logmel_front_end_against_scipy_stft_and_slaney_landmarks():
    """librosa is absent, so the restated front end (mr_gan.py:45-47) is pinned piecewise: the framing / window / FFT against
    scipy.signal.stft (an independent implementation; centred frames = reflect padding, periodic Hann, hop 512), the mel
    scale against Slaney's published landmarks (linear 200/3 Hz per mel below 1 kHz, 27 mels per factor 6.4 above), the
    filters against their defining properties (triangles between neighbouring centres, area-normalised), and the dB
    conversion against its closed form."""
    import scipy.signal as ss
    from mr_gan_b200 import realdata
    rng = np.random.default_rng(1)
    y = rng.standard_normal(9600)                                         # 0.2 s at 48 kHz, processdata.py:12
    n_fft, hop = 2048, 512
    win = ss.get_window('hann', n_fft, fftbins=True)
    _, _, Z = ss.stft(np.pad(y, n_fft // 2, mode='reflect'), fs=48000, window=win, nperseg=n_fft, noverlap=n_fft - hop,
                      boundary=None, padded=False)
    P = np.abs(Z * win.sum()) ** 2                                        # undo scipy's spectrum scaling
    S = realdata.melspectrogram(y)
    assert S.shape == (128, 19)
    np.testing.assert_allclose(S, realdata.mel_filterbank() @ P, rtol=1e-10, atol=1e-12 * S.max())
    np.testing.assert_allclose(realdata._hz_to_mel([200.0 / 3, 1000.0, 6400.0]), [1.0, 15.0, 42.0], rtol=1e-12)
    np.testing.assert_allclose(realdata._mel_to_hz([1.0, 15.0, 42.0]), [200.0 / 3, 1000.0, 6400.0], rtol=1e-12)
    fb = realdata.mel_filterbank()
    edges = realdata._mel_to_hz(np.linspace(0.0, realdata._hz_to_mel(24000.0), 130))
    hz = np.arange(1025) * 48000 / 2048.0
    for m in (40, 90, 127):                                               # wide filters: many FFT bins per triangle
        tri = np.interp(hz, edges[m:m + 3], [0.0, 1.0, 0.0], left=0.0, right=0.0) * 2.0 / (edges[m + 2] - edges[m])
        np.testing.assert_allclose(fb[m], tri, atol=1e-12)
        assert abs(fb[m].sum() * 48000 / 2048.0 - 1.0) < 0.02              # unit area in Hz
    L = realdata.logamplitude(S)
    np.testing.assert_allclose(L, np.maximum(10 * np.log10(np.maximum(S, 1e-10) / S.max()), -80.0), atol=1e-9)


def test_real_data_loader_and_librosa_free_logmel(tmp_path):
    """dataset() on files in the processed-pickle format of processdata.py:91 (Python-2 protocol), and the numpy
    restatement of librosa's melspectrogram / logamplitude (shape, scale and peak-position properties)."""
    import pickle
    from mr_gan_b200 import realdata
    rng = np.random.default_rng(0)
    fb = realdata.mel_filterbank()
    assert fb.shape == (128, 1025) and (fb >= 0).all() and (fb.sum(axis=1) > 0).all()
    centers = fb.argmax(axis=1)
    assert (np.diff(centers) >= 0).all()                                  # monotone filter centres
    sr, n = 48000, 9600                                                   # 0.2 s window, processdata.py:12
    tone = np.sin(2 * np.pi * 3000.0 * np.arange(n) / sr)
    S = realdata.melspectrogram(tone)
    assert S.shape == (128, 1 + n // 512)                                 # 128 x 19 -> 2432 features (SURVEY.md 8)
    peak_hz = (np.arange(1025) * sr / 2048.0)[fb[S[:, 9].argmax()].argmax()]
    assert abs(peak_hz - 3000.0) < 150.0
    L = realdata.logamplitude(S)
    assert L.max() == 0.0 and L.min() >= -80.0
    # tiny fake "MREO" set: 6 materials x 2 objects x 3 pokes, 0.1 s force/temperature, 0.05 s contact
    for material in model.MATERIALS:
        data = {}
        for o in range(2):
            data["%s_obj%d" % (material, o)] = {
                'temperature': [list(rng.standard_normal(10)) for _ in range(3)],
                'force0': [list(rng.standard_normal(10)) for _ in range(3)],
                'force1': [list(rng.standard_normal(10)) for _ in range(3)],
                'contact': [list(rng.standard_normal(2400)) for _ in range(3)]}
        with open(realdata.processed_path(str(tmp_path), material, 0.1, 0.05), 'wb') as f:
            pickle.dump(data, f, protocol=2)
    widths = {0: 20, 1: 10, 2: 30, 3: 640, 4: 650, 5: 670, 6: 660}
    for mod, w in widths.items():
        X, y = mg.dataset(modalities=mod, forcetempTime=0.1, contactmicTime=0.05, data_dir=str(tmp_path))
        assert X.shape == (36, w) and list(np.bincount(y)) == [6] * 6
        assert w == synthetic.feature_width(mod, 0.1, 0.05)               # the synthetic generator has the same layout
    objs = mg.dataset(modalities=2, forcetempTime=0.1, contactmicTime=0.05, leaveObjectOut=True, data_dir=str(tmp_path))
    assert len(objs) == 12 and all(o['x'].shape == (3, 30) for o in objs.values())
