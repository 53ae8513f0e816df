"""ORACLE (test infrastructure only) -- restatement of the RBF C-SVC that mr_svm.py:106 fits
(sklearn's libsvm ``SVC(kernel='rbf', C)``) in NumPy, step for step as the CUDA path computes it.

Specification: the libsvm source shipped with sklearn, ``sklearn/svm/src/libsvm/svm.cpp``:
  kernel       kernel_rbf, svm.cpp:346-348; stored as float (Qfloat, svm.cpp:79), QD = K(i, i) = 1 in double
  solver       Solver::Solve, svm.cpp:666-943, without shrinking (which changes only the speed); alpha = 0, G = p = -1
  working set  select_working_set, svm.cpp:946-1043 (second-order rule, TAU = 1e-12, ties: the LAST index wins)
  bias         calculate_rho, svm.cpp:1126-1162
  prediction   svm_predict_values, svm.cpp:2865-2897 (one-vs-one vote, the first class with most votes wins)
One-vs-one: the 15 pairs (a < b) in order (0,1), (0,2), ..., (4,5); a pair's problem is the rows of class a (y = +1)
followed by those of class b (y = -1), in row order.  Never imported by the product path.
"""
import numpy as np

TAU = 1e-12


def rbf(A, B, gamma):
    """kernel_rbf in double: exp(-gamma (|a|^2 + |b|^2 - 2 a.b)), svm.cpp:346-348."""
    A, B = np.asarray(A, np.float64), np.asarray(B, np.float64)
    na, nb = (A * A).sum(1), (B * B).sum(1)
    return np.exp(-gamma * (na[:, None] + nb[None, :] - 2.0 * (A @ B.T)))


def pairs(n_classes):
    return [(a, b) for a in range(n_classes) for b in range(a + 1, n_classes)]


def solve(Kf, y, C=1.0, eps=1e-3, max_iter=None):
    """Solver::Solve for a C-SVC sub-problem.  Kf: the sub-problem's kernel matrix as stored (float32), y: +-1.
    Returns (alpha, rho, n_iter, hit_cap)."""
    n = len(y)
    y = np.asarray(y, np.float64)
    Q = (y[:, None] * y[None, :]) * np.asarray(Kf, np.float32).astype(np.float64)   # Qfloat -> double, exact
    QD = np.ones(n)
    alpha, G = np.zeros(n), -np.ones(n)
    cap = max(10 ** 7, 100 * n) if max_iter is None else max_iter
    it = 0
    pos = y > 0
    while True:
        if it >= cap:
            return alpha, _rho(alpha, G, y, C), it, True
        upper, lower = alpha >= C, alpha <= 0
        # i: argmax over I_up of -y G (scan with >=: the last maximum wins)
        cand_i = np.where(pos, ~upper, ~lower)
        Gmax, i = -np.inf, -1
        if cand_i.any():
            v = np.where(cand_i, -y * G, -np.inf)
            Gmax = v.max()
            i = int(np.nonzero(cand_i & (v == Gmax))[0][-1])
        # j: Gmax2 = max over I_low of y G; argmin obj_diff over I_low with grad_diff > 0 (<=: the last minimum wins)
        cand_j = np.where(pos, ~lower, ~upper)
        Gmax2 = np.max(np.where(cand_j, y * G, -np.inf)) if cand_j.any() else -np.inf
        j = -1
        if i >= 0:
            grad_diff = Gmax + y * G
            quad = QD[i] + QD - 2.0 * y[i] * y * Q[i]      # = QD_i + QD_j - 2 K_ij in both branches of svm.cpp:997/1021
            quad = np.where(quad > 0, quad, TAU)
            obj = -(grad_diff * grad_diff) / quad
            ok = cand_j & (grad_diff > 0)
            if ok.any():
                m = np.where(ok, obj, np.inf).min()
                j = int(np.nonzero(ok & (obj == m))[0][-1])
        if Gmax + Gmax2 < eps or j == -1:
            break
        it += 1
        ai, aj = alpha[i], alpha[j]
        if y[i] != y[j]:                                   # svm.cpp:770-812
            quad = QD[i] + QD[j] + 2 * Q[i, j]
            if quad <= 0:
                quad = TAU
            delta = (-G[i] - G[j]) / quad
            diff = ai - aj
            ni, nj = ai + delta, aj + delta
            if diff > 0:
                if nj < 0:
                    nj, ni = 0.0, diff
            elif ni < 0:
                ni, nj = 0.0, -diff
            if diff > 0:                                   # C_i - C_j = 0
                if ni > C:
                    ni, nj = C, C - diff
            elif nj > C:
                nj, ni = C, C + diff
        else:                                              # svm.cpp:813-855
            quad = QD[i] + QD[j] - 2 * Q[i, j]
            if quad <= 0:
                quad = TAU
            delta = (G[i] - G[j]) / quad
            s = ai + aj
            ni, nj = ai - delta, aj + delta
            if s > C:
                if ni > C:
                    ni, nj = C, s - C
            elif nj < 0:
                nj, ni = 0.0, s
            if s > C:
                if nj > C:
                    nj, ni = C, s - C
            elif ni < 0:
                ni, nj = 0.0, s
        alpha[i], alpha[j] = ni, nj
        dai, daj = ni - ai, nj - aj
        G += Q[i] * dai + Q[j] * daj                       # svm.cpp:862-865
    return alpha, _rho(alpha, G, y, C), it, False


def _rho(alpha, G, y, C):
    """calculate_rho, svm.cpp:1126-1162 (sequential sum over the free variables)."""
    ub, lb, s, nfree = np.inf, -np.inf, 0.0, 0
    for a, g, yy in zip(alpha, G, y):
        yG = yy * g
        if a >= C:
            if yy < 0:
                ub = min(ub, yG)
            else:
                lb = max(lb, yG)
        elif a <= 0:
            if yy > 0:
                ub = min(ub, yG)
            else:
                lb = max(lb, yG)
        else:
            nfree += 1
            s += yG
    return s / nfree if nfree > 0 else (ub + lb) / 2


def fit_predict(x_lab, y_lab, x_test, gamma, C=1.0, eps=1e-3, n_classes=6):
    """One-vs-one fit on class-major labeled rows and prediction of x_test.
    Returns dict(dec [n_test, n_pairs], pred [n_test], n_iter [n_pairs], rho [n_pairs])."""
    y_lab = np.asarray(y_lab)
    Kf = rbf(x_lab, x_lab, gamma).astype(np.float32)
    Kt = rbf(x_test, x_lab, gamma)                         # svm_predict_values evaluates the kernel in double
    P = pairs(n_classes)
    dec = np.zeros((len(x_test), len(P)))
    n_iter, rhos = np.zeros(len(P), np.int64), np.zeros(len(P))
    for p, (a, b) in enumerate(P):
        rows = np.concatenate([np.nonzero(y_lab == a)[0], np.nonzero(y_lab == b)[0]])
        yy = np.where(y_lab[rows] == a, 1.0, -1.0)
        alpha, rho, it, _ = solve(Kf[np.ix_(rows, rows)], yy, C, eps)
        dec[:, p] = Kt[:, rows] @ (alpha * yy) - rho
        n_iter[p], rhos[p] = it, rho
    votes = np.zeros((len(x_test), n_classes), np.int64)
    for p, (a, b) in enumerate(P):
        votes[:, a] += dec[:, p] > 0
        votes[:, b] += dec[:, p] <= 0
    return dict(dec=dec, pred=np.argmax(votes, axis=1), n_iter=n_iter, rho=rhos)
