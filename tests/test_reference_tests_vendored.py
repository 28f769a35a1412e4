"""The reference's tests are vendored byte for byte (tests/reference_tests/) and run on the B200 through the shims;
here (CPU): the copies are intact, and the oct2py shim really executes the vendored .m files."""
import hashlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RT = os.path.join(ROOT, "tests", "reference_tests")


def _sha(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def test_vendored_files_match_their_checksums_and_the_reference():
    # sha256sums.txt holds the digests of the reference's own tests/ files (nrontsis/PILCO)
    lines = [ln.rstrip("\n") for ln in open(os.path.join(RT, "sha256sums.txt")) if ln.strip()]
    assert len(lines) == 16                                   # 5 test files + 10 .m files + license.txt
    for ln in lines:
        digest, rel = ln.split("  ", 1)
        assert _sha(os.path.join(RT, rel)) == digest, "vendored copy differs from the reference's tests/" + rel
    names = sorted(f for f in os.listdir(RT) if f.startswith("test_") and f.endswith(".py"))
    assert names == ["test_cascade.py", "test_controllers.py", "test_predictions.py", "test_rewards.py",
                     "test_sparse_predictions.py"]


def test_oct2py_shim_executes_the_vendored_m_files():
    """The shim runs gp0.m / reward.m / pred.m themselves (oracle/mrun.py); the independent transcription
    oracle/matlab_port.py agrees to ~1e-12 -- two routes to the same numbers."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "shims"))
    import oct2py
    from oracle import matlab_port as mp
    from util import hyp_of
    assert os.path.samefile(oct2py._MDIR, os.path.join(RT, "Matlab Code")) and not oct2py._USE_PORT
    octave = oct2py.Oct2Py()
    np.random.seed(0)
    d, k = 3, 2
    X0 = np.random.rand(40, d); A = np.random.rand(d, k)
    Y0 = np.sin(X0).dot(A) + 1e-3 * (np.random.rand(40, k) - 0.5)
    m = np.random.rand(1, d); s = np.random.rand(d, d); s = s.dot(s.T)
    ell, sf2, sn2 = 1.0 + np.random.rand(k, d), 0.5 + np.random.rand(k), 1e-3 * np.ones(k)
    gpmodel = oct2py.io.Struct()
    gpmodel.hyp = hyp_of(ell, sf2, sn2); gpmodel.inputs = X0; gpmodel.targets = Y0
    M, S, V = octave.gp0(gpmodel, m.T, s, nout=3)
    Mp, Sp, Vp = mp.gp0(dict(hyp=gpmodel.hyp, inputs=X0, targets=Y0), m.T, s)
    for a, b in ((M, Mp), (S, Sp), (V, Vp)):
        np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=1e-9, atol=1e-12)
    mr = np.random.rand(1, 2); sr = np.random.rand(2, 2); sr = sr.dot(sr.T)
    muR, _, _, sR = octave.reward(mr.T, sr, np.zeros((2, 1)), np.eye(2), nout=4)
    ref = mp.reward(mr.T, sr, np.zeros((2, 1)), np.eye(2))
    np.testing.assert_allclose(np.asarray(muR), np.asarray(ref[0]), rtol=1e-12)
    np.testing.assert_allclose(np.asarray(sR), np.asarray(ref[3]), rtol=1e-10)
    with pytest.raises(AttributeError):
        octave.no_such_function
