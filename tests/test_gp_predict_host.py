"""pilco_gp_predict without a GPU: the GPflow oracle against the factor identity the kernel evaluates, the ABI's argument
validation, the workspace bound (K* is never materialised on the diagonal path) and the SASS of the fused kernel."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from gp_predict_oracle import factor_predict_f, predict_f
from oracle import python_port as pp
from pilco_b200 import _lib
from pilco_b200._lib import lib
from util import make_gp_problem

OK, ERR_NULL, ERR_DIM, ERR_WS, ERR_UNSUP = 0, -1, -2, -3, -6
FAKE = 0x10000          # never dereferenced: only rejecting calls (and B = 0 no-ops) are made
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "pilco_b200", "libpilco_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def _var_bar(iK, sf2):
    """The quadratic form k*' iK k* cancels against sf2 and goes through an explicit inverse, so its round-off grows with
    the condition number of iK: 1e-12 sf2 for a well-conditioned model, 1e-15 cond(iK) sf2 beyond (cond = 6e4 and
    6e5 for the two noise levels below)."""
    return np.array([max(1e-12, 1e-15 * np.linalg.cond(iK[e])) * sf2[e] for e in range(len(sf2))])


@pytest.mark.parametrize("sn2", [1e-2, 1e-3])
def test_oracle_matches_factor_identity_exact_gp(sn2):
    X, Y, ell, sf2, _ = make_gp_problem(400, 5, 3, seed=11)
    sn = sn2 * np.ones(3)
    Xnew = np.random.RandomState(12).rand(64, 5) * 1.2 - 0.1
    iK, beta = pp.calculate_factorizations(X, Y, ell, sf2, sn)
    m0, v0 = predict_f(X, Y, ell, sf2, sn, Xnew)
    m1, v1 = factor_predict_f(X, ell, sf2, iK, beta, Xnew)
    assert np.max(np.abs(m1 - m0)) <= 1e-12 * np.max(np.abs(m0))
    assert np.all(np.max(np.abs(v1 - v0), axis=0) <= _var_bar(iK, sf2))


@pytest.mark.parametrize("sn2", [1e-2, 1e-3])
def test_oracle_matches_factor_identity_fitc(sn2):
    X, Y, ell, sf2, _ = make_gp_problem(400, 5, 3, seed=13)
    sn = sn2 * np.ones(3)
    Z = X[np.random.RandomState(14).choice(400, 40, replace=False)]
    Xnew = np.random.RandomState(15).rand(64, 5)
    iK, beta = pp.fitc_factorizations(X, Z, Y, ell, sf2, sn)
    m0, v0 = predict_f(X, Y, ell, sf2, sn, Xnew, Z=Z)
    m1, v1 = factor_predict_f(Z, ell, sf2, iK, beta, Xnew)
    assert np.max(np.abs(m1 - m0)) <= 1e-12 * np.max(np.abs(m0))
    assert np.all(np.max(np.abs(v1 - v0), axis=0) <= _var_bar(iK, sf2))


def test_oracle_full_cov_diagonal_is_the_diagonal_path():
    X, Y, ell, sf2, sn2 = make_gp_problem(100, 4, 2, seed=16)
    Xnew = np.random.RandomState(17).rand(20, 4)
    for Z in (None, X[:30]):
        m, v = predict_f(X, Y, ell, sf2, sn2, Xnew, Z=Z)
        mc, c = predict_f(X, Y, ell, sf2, sn2, Xnew, Z=Z, full_cov=True)
        assert np.array_equal(m, mc)
        assert np.max(np.abs(np.diagonal(c, axis1=1, axis2=2).T - v)) <= 1e-13


def _gp(n=50, D=4, E=3, mode=0, iK=FAKE, ldk=64):
    g = _lib.GpModel()
    g.n, g.D, g.E, g.mode = n, D, E, mode
    g.X = g.ell = g.sf2 = g.beta = FAKE
    g.iK, g.ldk = iK, ldk
    return g


def test_gp_predict_argument_validation():
    f = lambda g, B=4, mean=FAKE, var=FAKE, cov=None, ws=None, wsb=0: lib.pilco_gp_predict(
        C.byref(g) if g is not None else None, B, FAKE, mean, var, cov, ws, wsb, None)
    assert f(None) == ERR_NULL
    assert f(_gp(iK=None)) == ERR_NULL                                      # var of a model without iK (mode 1 / RBF)
    assert f(_gp(iK=None), var=None, cov=FAKE, ws=FAKE, wsb=1 << 30) == ERR_NULL
    g = _gp(); g.X_bs = 200
    assert f(g) == ERR_DIM                                                  # batched models are rejected
    g = _gp(); g.beta_bs = 150
    assert f(g) == ERR_DIM
    assert f(_gp(D=17)) == ERR_DIM                                          # D > PILCO_MAX_D
    assert f(_gp(E=0)) == ERR_DIM and f(_gp(E=17)) == ERR_DIM
    assert f(_gp(ldk=32)) == ERR_DIM                                        # ldk < pilco_pad_n(n)
    assert f(_gp(), B=-1) == ERR_DIM
    assert f(_gp(), cov=FAKE, wsb=0, ws=FAKE) == ERR_WS                       # full_cov needs its workspace
    need = lib.pilco_gp_predict_workspace_bytes(50, 4, 3, 4, 1)
    assert need > 0 and f(_gp(), cov=FAKE, ws=FAKE, wsb=need - 8) == ERR_WS
    assert f(_gp(), mean=None, var=None) == ERR_NULL                        # nothing requested
    assert f(_gp(n=5000, ldk=5056)) == ERR_UNSUP                            # K* row block beyond shared memory
    assert f(_gp(), B=0) == OK                                               # no-op: nothing is enqueued
    assert f(_gp(iK=None), B=0, var=None) == OK


def test_gp_predict_workspace_does_not_hold_kstar():
    assert lib.pilco_gp_predict_workspace_bytes(300, 12, 10, 100000, 0) < 100000 * 300 * 10 * 8
    assert lib.pilco_gp_predict_workspace_bytes(300, 12, 10, 100000, 0) == 0
    assert lib.pilco_gp_predict_workspace_bytes(300, 12, 10, 64, 1) == 2 * 10 * 64 * 320 * 8
    assert lib.pilco_gp_predict_workspace_bytes(300, 17, 10, 64, 0) == 0


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_gp_predict_kernel_sass():
    """Every instantiation of the fused kernel (8, 16, 32 points per CTA) runs the quadratic form on DMMA.8x8x4, uses the
    table exp (no MUFU.EX2) and keeps everything in registers and shared memory (no local memory); sm_100a cubin."""
    out = subprocess.run([CUOBJDUMP, "-sass", LIB], capture_output=True, text=True, timeout=600).stdout
    funcs, name, arch = {}, None, None
    for line in out.splitlines():
        m = re.search(r"arch = (sm_\w+)", line)
        if m:
            arch = m.group(1)
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1) if "gp_predict_kernel" in m.group(1) else None
            if name:
                funcs[name] = [arch]
        elif name:
            funcs[name].append(line)
    assert len(funcs) == 3, sorted(funcs)
    for name, lines in funcs.items():
        text = "\n".join(lines[1:])
        assert lines[0] == "sm_100a", (name, lines[0])
        assert "DMMA.8x8x4" in text, name
        assert not re.search(r"\b(STL|LDL)\b", text), "local memory traffic in %s" % name
        assert "MUFU.EX2" not in text, name
