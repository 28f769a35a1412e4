"""Generate tests/golden/*.npz by EXECUTING the reference's MATLAB oracle files
(tests/reference_tests/Matlab Code/*.m) with oracle/mrun.py, on the seeded recipes of the reference's tests
(tests/test_predictions.py, test_sparse_predictions.py, test_controllers.py, test_rewards.py,
test_cascade.py) plus the BASELINE metric shape.  Hyper-parameters are fixed seeded values (the reference
feeds whatever its optimisers return to the oracle; trajectories are not pinned, SURVEY.md section 4).

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import mrun            # noqa: E402
from util import hyp_of            # noqa: E402


def recipe_data(n, d, k, seed=0):
    np.random.seed(seed)
    X0 = np.random.rand(n, d)
    A = np.random.rand(d, k)
    Y0 = np.sin(X0).dot(A) + 1e-3 * (np.random.rand(n, k) - 0.5)
    m = np.random.rand(1, d)
    s = np.random.rand(d, d)
    s = s.dot(s.T)
    return X0, Y0, m, s


def hypers(k, d, seed, noise=1e-3):
    rng = np.random.RandomState(seed)
    return 1.0 + rng.rand(k, d), 0.5 + rng.rand(k), noise * (1.0 + rng.rand(k))


def main():
    out = {}
    # --- gp0 : tests/test_predictions.py recipe (two data sets) + metric shape -------------------------
    X0, Y0, m, s = recipe_data(100, 3, 2)
    ell, sf2, sn2 = hypers(2, 3, 1)
    for tag, X in (("a", X0), ("b", 5 * np.random.RandomState(7).rand(100, 3))):
        M, S, V = mrun.run("gp0", dict(hyp=hyp_of(ell, sf2, sn2), inputs=X, targets=Y0), m.T, s, nout=3)
        out["gp0_" + tag] = dict(X=X, Y=Y0, ell=ell, sf2=sf2, sn2=sn2, m=m, s=s, M=M, S=S, V=V)
    Xb, Yb, mb, sb = recipe_data(300, 12, 10, seed=3)
    ellb, sf2b, sn2b = hypers(10, 12, 4, noise=1e-2)
    M, S, V = mrun.run("gp0", dict(hyp=hyp_of(ellb, sf2b, sn2b), inputs=Xb, targets=0.1 * Yb), mb.T, 0.05 * sb, nout=3)
    out["gp0_metric"] = dict(X=Xb, Y=0.1 * Yb, ell=ellb, sf2=sf2b, sn2=sn2b, m=mb, s=0.05 * sb, M=M, S=S, V=V)
    # --- gp1 : tests/test_sparse_predictions.py ----------------------------------------------------------
    Z = np.random.RandomState(5).rand(30, 3)
    M, S, V = mrun.run("gp1", dict(hyp=hyp_of(ell, sf2, sn2), inputs=X0, targets=Y0, induce=Z), m.T, s, nout=3)
    out["gp1"] = dict(X=X0, Y=Y0, Z=Z, ell=ell, sf2=sf2, sn2=sn2, m=m, s=s, M=M, S=S, V=V)
    # --- gp2 : tests/test_controllers.py::test_rbf --------------------------------------------------------
    ellc = 1.0 + 0.3 * np.random.RandomState(6).rand(2, 3)
    hyp = hyp_of(ellc, np.ones(2), 1e-4 * np.ones(2))
    M, S, V = mrun.run("gp2", dict(hyp=hyp, inputs=X0, targets=Y0), m.T, s, nout=3)
    out["gp2"] = dict(X=X0, Y=Y0, ell=ellc, m=m, s=s, M=M, S=S, V=V)
    # --- conlin / gSin / reward -----------------------------------------------------------------------------
    rng = np.random.RandomState(8)
    W, b = rng.rand(2, 3), rng.rand(1, 2)
    M, S, V = mrun.run("conlin", dict(p=dict(w=W, b=b.T)), m.T, s, nout=3)
    out["conlin"] = dict(W=W, b=b, m=m, s=s, M=M, S=S, V=V)
    M, S, C = mrun.run("gSin", m.T, s, 7.0, nout=3)
    out["gSin"] = dict(m=m, s=s, e=np.array(7.0), M=M, S=S, C=C)
    for kdim in (2, 5):
        mr = rng.rand(1, kdim); sr = rng.rand(kdim, kdim); sr = sr.dot(sr.T)
        Wr = np.eye(kdim) if kdim == 2 else np.diag(0.5 + rng.rand(kdim))
        tr = np.zeros((1, kdim)) if kdim == 2 else rng.rand(1, kdim)
        muR, dm, dS, sR = mrun.run("reward", mr.T, sr, tr.T, Wr, nout=4)
        out["reward_%d" % kdim] = dict(m=mr, s=sr, W=Wr, t=tr, muR=muR, dmuRdm=dm, dmuRdS=dS, sR=sR)
    # --- pred / propagate : tests/test_cascade.py --------------------------------------------------------------
    np.random.seed(0)
    d, k, H = 2, 1, 10
    X0 = np.random.rand(100, d + k)
    A = np.random.rand(d + k, d)
    Y0 = np.sin(X0).dot(A) + 1e-3 * (np.random.rand(100, d) - 0.5)
    ell, sf2, sn2 = hypers(d, d + k, 9)
    W, b, e = rng.rand(k, d), rng.rand(1, k), np.array([[10.0]])
    m = np.random.rand(1, d); s = np.random.rand(d, d); s = s.dot(s.T)
    plant = dict(angi=np.zeros((0, 0)), poli=np.arange(d) + 1.0, dyni=np.arange(d) + 1.0, difi=np.arange(d) + 1.0)
    Mt, St = mrun.run("pred", dict(p=dict(w=W, b=b.T), maxU=e), plant,
                      dict(hyp=hyp_of(ell, sf2, sn2), inputs=X0, targets=Y0), m.T, s, float(H), nout=2)
    out["pred"] = dict(X=X0, Y=Y0, ell=ell, sf2=sf2, sn2=sn2, W=W, b=b, e=e, m=m, s=s, H=np.array(H), Mtraj=Mt, Straj=St)
    for name, d_ in out.items():
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **{k_: np.asarray(v) for k_, v in d_.items()})
        print("wrote", name, {k_: np.asarray(v).shape for k_, v in d_.items() if k_ in ("M", "S", "V", "Mtraj", "Straj", "muR")})


if __name__ == "__main__":
    main()
