"""numpy restatement of GPflow 2's predictive at deterministic inputs, written from the formulas (GPflow itself is not a
dependency): ``GPR.predict_f`` in its Cholesky form and ``GPRFITC.predict_f`` in its ``common_terms`` form (jitter 1e-6
on Kuu), one output at a time.  The oracle of pilco_gp_predict (tests/test_gp_predict_host.py, tests/test_gpu_predict.py).
"""
import numpy as np
from scipy.linalg import cholesky, solve_triangular

JITTER = 1e-6


def se_ard(X1, X2, ell, sf2):
    """gpflow.kernels.SquaredExponential.K for one output: sf2 exp(-0.5 |(x - x') / ell|^2)"""
    d = (X1[:, None, :] - X2[None, :, :]) / ell
    return sf2 * np.exp(-0.5 * np.sum(d * d, axis=-1))


def gpr_predict_f(X, y, ell, sf2, sn2, Xnew, full_cov=False):
    """GPR.predict_f: L = chol(K + sn2 I), A = L^-1 K(X, Xnew); mean = A' L^-1 y; var = k** - A'A.
    -> mean [B], var [B] (or cov [B,B])"""
    L = cholesky(se_ard(X, X, ell, sf2) + sn2 * np.eye(X.shape[0]), lower=True)
    A = solve_triangular(L, se_ard(X, Xnew, ell, sf2), lower=True)
    mean = A.T @ solve_triangular(L, y, lower=True)
    if full_cov:
        return mean, se_ard(Xnew, Xnew, ell, sf2) - A.T @ A
    return mean, sf2 - np.sum(A * A, axis=0)


def gprfitc_predict_f(X, y, Z, ell, sf2, sn2, Xnew, full_cov=False):
    """GPRFITC.predict_f (common_terms): Luu = chol(Kuu + jitter I), V = Luu^-1 Kuf, nu = diag(Kff) - diag(V'V) + sn2,
    L = chol(I + V diag(1/nu) V'), gamma = L^-1 V (y / nu);  at Xnew: w = Luu^-1 Kus, t = L^-1 w,
    mean = t' gamma, var = k** - w'w + t't.  -> mean [B], var [B] (or cov [B,B])"""
    M = Z.shape[0]
    Luu = cholesky(se_ard(Z, Z, ell, sf2) + JITTER * np.eye(M), lower=True)
    V = solve_triangular(Luu, se_ard(Z, X, ell, sf2), lower=True)
    nu = sf2 - np.sum(V * V, axis=0) + sn2
    L = cholesky(np.eye(M) + (V / nu) @ V.T, lower=True)
    gamma = solve_triangular(L, V @ (y / nu), lower=True)
    w = solve_triangular(Luu, se_ard(Z, Xnew, ell, sf2), lower=True)
    t = solve_triangular(L, w, lower=True)
    mean = t.T @ gamma
    if full_cov:
        return mean, se_ard(Xnew, Xnew, ell, sf2) - w.T @ w + t.T @ t
    return mean, sf2 - np.sum(w * w, axis=0) + np.sum(t * t, axis=0)


def predict_f(X, Y, ell, sf2, sn2, Xnew, Z=None, full_cov=False):
    """All E outputs: mean [B,E] and var [B,E] (or cov [E,B,B]); FITC over Z when given."""
    outs = [gpr_predict_f(X, Y[:, e], ell[e], sf2[e], sn2[e], Xnew, full_cov) if Z is None else
            gprfitc_predict_f(X, Y[:, e], Z, ell[e], sf2[e], sn2[e], Xnew, full_cov) for e in range(Y.shape[1])]
    mean = np.stack([o[0] for o in outs], axis=1)
    v = np.stack([o[1] for o in outs], axis=0 if full_cov else 1)
    return mean, v


def factor_predict_f(C, ell, sf2, iK, beta, Xnew):
    """The identity pilco_gp_predict evaluates, from (iK [E,n,n], beta [E,n]) over centres C:
    mean = K* beta, var = sf2 - rowsum((K* iK) o K*)."""
    E = ell.shape[0]
    Ks = [se_ard(Xnew, C, ell[e], sf2[e]) for e in range(E)]
    mean = np.stack([Ks[e] @ beta[e] for e in range(E)], axis=1)
    var = np.stack([sf2[e] - np.sum((Ks[e] @ iK[e]) * Ks[e], axis=1) for e in range(E)], axis=1)
    return mean, var
