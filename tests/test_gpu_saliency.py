"""GPU tier of the input gradients (mrgan_input_grad, mrgan_saliency): parity with the float64 reference in all three
precisions and in the LeakyReLU / Dropout variants, bitwise reproduction of the resident test set by new rows, the class
profiles against numpy, reproducibility and grouping independence, no side effect on anything the group computes later,
error codes, and the mr_nn CLI's --saliency flag."""
import json
import re

import numpy as np
import pytest

from mr_gan_b200 import _lib, mr_gan, mr_nn, synthetic
from mr_gan_b200.engine import FoldGroup, MrganError

import saliency_ref as R
from test_gpu_predict import K, NTE, NTR, _folds, _group, _svm_fit

pytestmark = pytest.mark.gpu


def _x_test(fg, i, D):
    return fg.debug_buffer(i, 51, NTE, D).astype(np.float64)      # the resident X_test as the kernels read it


def _params(fg, i):
    return [p.astype(np.float64) for p in fg.get_params(i, 0)]


# Norm-wise relative error ||g - ref|| / ||ref|| allowed in tf32 / f16: about twice the largest measured (see below).
GRAD_TOL = {"tf32": 1e-1, "f16": 1e-1}


@pytest.mark.parametrize("precision", ["fp32", "tf32", "f16"])
@pytest.mark.parametrize("model", ["gan", "nn"])
def test_input_grad_matches_reference(model, precision):
    """Heterogeneous group (D = 400 and 1200, n_test = 97) after one epoch, target = the predicted class: the gradients of
    the float64 reference on the weights read back.  fp32: max |error| <= 1e-5 of the fold's largest |g|; measured on a
    B200: 1.2e-6 (GAN) and 8.2e-7 (NN), accumulation order only.  tf32 / f16 (10-bit operand mantissas through six layers,
    and a pre-activation near zero whose ReLU mask flips moves a whole column of the chain): norm-wise, measured at most
    3.2e-2 / 2.5e-2 (GAN) and 5.5e-2 / 5.5e-2 (NN) in tf32 / f16."""
    folds = _folds((400, 1200))
    errs = []
    with _group(model, precision, folds) as fg:
        for i, f in enumerate(folds):
            g = fg.input_grad(i)
            assert g.shape == (NTE, f['D']) and g.dtype == np.float32
            pred = fg.predict(i)[0]
            ref = R.input_grad(_params(fg, i), _x_test(fg, i, f['D']), pred)
            if precision == "fp32":
                errs.append(np.abs(g - ref).max() / np.abs(ref).max())
            else:
                errs.append(np.linalg.norm(g - ref) / np.linalg.norm(ref))
    print("MEASURED %s %s %s" % (model, precision, ["%.3g" % e for e in errs]))
    assert max(errs) <= (1e-5 if precision == "fp32" else GRAD_TOL[precision]), errs


@pytest.mark.parametrize("variant", ["leaky", "dropout"])
def test_input_grad_of_the_variants(variant):
    """LeakyReLU(0.3): the slope of the forward; Dropout(0.3): phase 0 has no dropout, so the gradient is the plain ReLU
    net's (fp32, GAN, after one epoch)."""
    folds = _folds((400,))
    hyper = dict(hidden_act=1, leaky_alpha=0.3) if variant == "leaky" else dict(dropout=0.3)
    f = folds[0]
    with FoldGroup([(f['D'], NTR, NTE, f['seed'])], model='gan', precision='fp32', batch=50, **hyper) as fg:
        fg.set_params(0, 1, f['pG'])
        fg.set_params(0, 0, f['pD'])
        fg.load_fold(0, f['xtr'], f['ytr'], f['xte'], f['yte'])
        fg.train_epoch(*[f['idx'][0][s][None] for s in range(3)])
        g = fg.input_grad(0)
        ref = R.input_grad(_params(fg, 0), _x_test(fg, 0, f['D']), fg.predict(0)[0], alpha=0.3 if variant == "leaky" else 0.0)
        err = np.abs(g - ref).max() / np.abs(ref).max()
        print("MEASURED variant %s max-rel %.3g" % (variant, err))
        assert err <= 1e-5, err


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_rows_targets_and_profile(precision):
    """New rows reproduce the resident path bitwise (n = 1, odd, n_test, > n_test); an explicit target = the predicted class
    equals target=None bitwise; saliency() is the class means of |input_grad(target=y_test)|, reproducible bitwise."""
    folds = _folds((400, 1200))
    with _group('gan', precision, folds) as fg:
        prof = fg.saliency()
        assert [p.shape for p in prof] == [(K, 400), (K, 1200)] and all(p.dtype == np.float32 for p in prof)
        for i, f in enumerate(folds):
            g = fg.input_grad(i)
            pred = fg.predict(i)[0]
            np.testing.assert_array_equal(fg.input_grad(i, target=pred), g)
            xt = fg.debug_buffer(i, 51, NTE, f['D'])
            for n in (1, 7, NTE, NTE + 13):
                idx = np.arange(n) % NTE
                np.testing.assert_array_equal(fg.input_grad(i, x=xt[idx]), g[idx])
                np.testing.assert_array_equal(fg.input_grad(i, x=xt[idx], target=pred[idx]), g[idx])
            gt = np.abs(fg.input_grad(i, target=f['yte']).astype(np.float64))
            want = np.stack([gt[f['yte'] == c].mean(axis=0) for c in range(K)])
            np.testing.assert_allclose(prof[i], want, rtol=1e-6, atol=0)
        again = fg.saliency()
        for a, b in zip(prof, again):
            np.testing.assert_array_equal(a, b)


def test_profile_grouping_independent_and_empty_class():
    folds = _folds((400, 1200))
    folds[1]['yte'] = np.where(folds[1]['yte'] == K - 1, 0, folds[1]['yte']).astype(np.int32)     # no test row of the last class
    with _group('gan', 'f16', folds, epochs=2) as fg:
        both = fg.saliency()
    assert not both[1][K - 1].any() and both[1][:K - 1].all()
    for i in range(2):
        with _group('gan', 'f16', [folds[i]], epochs=2) as fg:
            np.testing.assert_array_equal(fg.saliency()[0], both[i])


def _idx(rng, epochs):
    return [np.stack([np.stack([rng.permutation(NTR) for _ in range(3)]) for _ in range(2)]).astype(np.int32) for _ in range(epochs)]


@pytest.mark.parametrize("model,precision", [("gan", "f16"), ("nn", "tf32")])
def test_no_side_effects(model, precision):
    """A group that calls input_grad and saliency between epochs, and once with an epoch pending, computes bitwise what its
    twin that never calls them computes: pending and next epoch statistics, parameters, Adam state, eval, predict, confusion."""
    folds = _folds((400, 1200))
    idx = _idx(np.random.default_rng(9), 3)

    def run(probe):
        out = []
        with _group(model, precision, folds) as fg:
            for e in range(3):
                if probe:
                    fg.input_grad(0)
                    fg.input_grad(1, x=folds[1]['xte'][:5], target=np.arange(5) % K)
                    fg.saliency()
                if model == 'gan':
                    fg.train_epoch(idx[e][:, 0], idx[e][:, 1], idx[e][:, 2], wait=False)
                else:
                    fg.nn_train_epoch(idx[e][:, 0, :240], wait=False)
                if probe:
                    fg.saliency()
                    fg.input_grad(1)
                out.append(fg.epoch_result())
            for i in range(2):
                for net in ((0, 1) if model == 'gan' else (0,)):
                    out += fg.get_params(i, net) + [a for m in fg.get_adam(i, net) for a in m]
                out.append(np.array(fg.counters(i)))
                out += [np.float32(fg.eval(i)) if model == 'gan' else np.array(fg.nn_evaluate(i))] + list(fg.predict(i))
            out.append(fg.confusion())
        return out

    for a, b in zip(run(True), run(False)):
        np.testing.assert_array_equal(a, b)


def test_error_codes():
    ERR_ARG, ERR_STATE = -1, -4
    lib = _lib.load()
    x = np.zeros((NTE + 1, 16), np.float32)
    g = np.zeros((NTE + 1, 16), np.float32)
    prof = np.zeros((2, K, 16), np.float32)
    X, G, Pr = _lib.fptr(x), _lib.fptr(g), _lib.fptr(prof)
    tgt = np.zeros(NTE, np.int32)

    def T(v):
        tgt[:] = 0
        tgt[3] = v
        return _lib.iptr(tgt)

    folds = _folds((16, 16))
    with FoldGroup([(16, NTR, NTE, 0)]) as fg:                          # a GAN fold that is not loaded
        assert lib.mrgan_input_grad(fg._h, 0, None, NTE, None, G) == ERR_STATE
        assert lib.mrgan_saliency(fg._h, Pr) == ERR_STATE
    with _group('nn', 'fp32', folds[:1]) as fg:
        h = fg._h
        assert lib.mrgan_input_grad(h, 0, None, NTE, None, None) == ERR_ARG
        assert lib.mrgan_saliency(h, None) == ERR_ARG
        assert lib.mrgan_input_grad(h, 1, X, 1, None, G) == ERR_ARG and lib.mrgan_input_grad(h, -1, X, 1, None, G) == ERR_ARG
        assert lib.mrgan_input_grad(h, 0, X, 0, None, G) == ERR_ARG
        assert lib.mrgan_input_grad(h, 0, X, NTE + 1, None, G) == ERR_ARG
        assert lib.mrgan_input_grad(h, 0, None, 5, None, G) == ERR_ARG
        assert lib.mrgan_input_grad(h, 0, X, NTE, T(-1), G) == ERR_ARG
        assert lib.mrgan_input_grad(h, 0, None, NTE, T(K), G) == ERR_ARG
        assert lib.mrgan_input_grad(h, 0, X, NTE, T(K - 1), G) == 0
        assert lib.mrgan_input_grad(h, 0, None, NTE, None, G) == 0
        assert lib.mrgan_saliency(h, Pr) == 0
        with pytest.raises(ValueError):
            fg.input_grad(0, x=x[:, :15])
    with FoldGroup([(16, NTR, NTE, 0)], model='svm') as fg:             # an SVM handle before svm_fit
        fg.load_fold(0, folds[0]['xtr'], folds[0]['ytr'], folds[0]['xte'], folds[0]['yte'])
        assert lib.mrgan_input_grad(fg._h, 0, None, NTE, None, G) == ERR_STATE
        assert lib.mrgan_saliency(fg._h, Pr) == ERR_STATE
    fg, _ = _svm_fit([(2, 16, False)])                                  # ... and after
    with fg:
        n = fg.shapes[0][2]
        big = np.zeros((n, fg.shapes[0][0]), np.float32)
        assert lib.mrgan_input_grad(fg._h, 0, None, n, None, _lib.fptr(big)) == ERR_STATE
        with pytest.raises(MrganError, match="error -4"):
            fg.saliency()
    with FoldGroup([(16, NTR, NTE, 5)] * 2, batch=20) as fg:           # virtual ranks
        fg.dp_init_virtual(2)
        for r in range(2):
            fg.set_params(r, 0, folds[0]['pD']); fg.set_params(r, 1, folds[0]['pG'])
            fg.load_fold(r, folds[0]['xtr'], folds[0]['ytr'], folds[0]['xte'], folds[0]['yte'])
        assert lib.mrgan_input_grad(fg._h, 0, None, NTE, None, G) == ERR_STATE
        assert lib.mrgan_input_grad(fg._h, 0, X, 1, None, G) == ERR_STATE
        assert lib.mrgan_saliency(fg._h, Pr) == ERR_STATE


# ---------------------------------------------------------------- the mr_nn CLI end to end
def test_mr_nn_cli_saliency(capsys, tmp_path):
    base = ['--tables', '2', '--synthetic', '--seed', '0', '--epochs', '1']
    assert mr_nn.main(base) == 0
    plain = capsys.readouterr().out.splitlines()
    path = tmp_path / 'nn.npz'
    assert mr_nn.main(base + ['--saliency', str(path)]) == 0
    flagged = capsys.readouterr().out.splitlines()
    assert [line for line in flagged if not line.startswith('Saliency share:')] == plain     # unchanged and in order
    shares = [line for line in flagged if line.startswith('Saliency share:')]
    assert len(shares) == 14
    with np.load(str(path)) as z:
        index = json.loads(str(z['index']))
        arrays = {k: z[k] for k in z.files if k != 'index'}
    assert len(index) == len(arrays) == 84
    for rec in index:
        mod = mr_gan.MODALITIES.index(rec['modality'])
        assert arrays['job_%d' % rec['job_id']].shape == (K, {2: 1200, 5: 3632}[mod])
        assert rec['blocks'] == [[n, w] for n, w in synthetic.block_widths(mod)]
    for k, line in enumerate(shares):
        setting = index[6 * k:6 * k + 6]
        tot = np.sum([arrays['job_%d' % r['job_id']].astype(np.float64).sum(axis=0) for r in setting], axis=0)
        edges = np.cumsum([0] + [w for _, w in setting[0]['blocks']])
        mass = np.array([tot[a:b].sum() for a, b in zip(edges[:-1], edges[1:])])
        got = [float(v) for v in re.findall(r' (\d\.\d{3})', line)]
        assert got == [float('%.3f' % v) for v in mass / mass.sum()]
