"""Golden vectors produced by executing the reference's own MATLAB oracle files (tests/golden/make_golden.py,
oracle/mrun.py).  CPU part: both oracle transcriptions reproduce them (this is what pins the oracle);
GPU part: the device path through the C ABI reproduces them.  The reference's bar is rtol 1e-4 (2e-4 for the
cascade, 1e-7 for the reward); we hold fp64 tolerances written beside each assertion."""
import os

import numpy as np
import pytest

from util import scaled_err, hyp_of

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
load = lambda name: dict(np.load(os.path.join(G, name + ".npz")))


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["gp0_a", "gp0_b", "gp0_metric"])
def test_oracle_gp0_matches_reference_m_files(name):
    from oracle import matlab_port as mp, python_port as pp
    g = load(name)
    if name != "gp0_metric":          # the loop-form port is slow at N=300, E=10; the vectorised one covers it
        M, S, V = mp.gp0(dict(hyp=hyp_of(g["ell"], g["sf2"], g["sn2"]), inputs=g["X"], targets=g["Y"]), g["m"].T, g["s"])
        assert scaled_err(M, g["M"]) < 1e-11 and scaled_err(S, g["S"]) < 1e-9 and scaled_err(V, g["V"]) < 1e-10
    M, S, V = pp.predict_on_noisy_inputs(g["X"], g["Y"], g["ell"], g["sf2"], g["sn2"], g["m"], g["s"])
    assert scaled_err(M, g["M"].T) < 1e-10 and scaled_err(S, g["S"]) < 1e-8 and scaled_err(V, g["V"]) < 1e-9


def test_oracle_gp1_gp2_match_reference_m_files():
    from oracle import matlab_port as mp, python_port as pp
    g = load("gp1")
    M, S, V = mp.gp1(dict(hyp=hyp_of(g["ell"], g["sf2"], g["sn2"]), inputs=g["X"], targets=g["Y"], induce=g["Z"]), g["m"].T, g["s"])
    assert scaled_err(M, g["M"]) < 1e-9 and scaled_err(S, g["S"]) < 1e-8 and scaled_err(V, g["V"]) < 1e-9
    M, S, V = pp.sparse_predict_on_noisy_inputs(g["X"], g["Z"], g["Y"], g["ell"], g["sf2"], g["sn2"], g["m"], g["s"])
    assert scaled_err(M, g["M"].T) < 1e-8 and scaled_err(S, g["S"]) < 1e-7 and scaled_err(V, g["V"]) < 1e-8
    g = load("gp2")
    M, S, V = pp.rbf_action(g["X"], g["Y"], g["ell"], g["m"], g["s"], squash=False)
    assert scaled_err(M, g["M"].T) < 1e-10 and scaled_err(S, g["S"]) < 1e-9 and scaled_err(V, g["V"]) < 1e-9


def test_oracle_closed_forms_match_reference_m_files():
    from oracle import matlab_port as mp, python_port as pp
    g = load("conlin")
    M, S, V = pp.linear_action(g["W"], g["b"], g["m"], g["s"], squash=False)
    assert scaled_err(M, g["M"].T) < 1e-14 and scaled_err(S, g["S"]) < 1e-13 and scaled_err(V, g["V"]) < 1e-15
    g = load("gSin")
    M, S, C = pp.squash_sin(g["m"], g["s"], float(g["e"]))
    assert scaled_err(M, g["M"].T) < 1e-14 and scaled_err(S, g["S"]) < 1e-13 and scaled_err(C, g["C"]) < 1e-14
    for k in (2, 5):
        g = load("reward_%d" % k)
        mu, sR = pp.exponential_reward(g["m"], g["s"], g["W"], g["t"])
        assert abs(mu[0, 0] - g["muR"].item()) < 1e-14 and abs(sR[0, 0] - g["sR"].item()) < 1e-14
        from oracle import staged as st
        _, dm, dS = st.exp_reward_grad(g["m"][0], g["s"], g["W"], g["t"][0])
        assert scaled_err(dm, g["dmuRdm"][0]) < 1e-12 and scaled_err(dS, g["dmuRdS"]) < 1e-12   # reward.m:48-49


def test_oracle_cascade_matches_reference_m_files():
    from oracle import matlab_port as mp, python_port as pp
    g = load("pred")
    d = g["m"].shape[1]
    H = int(g["H"])
    plant = dict(angi=np.zeros(0), poli=np.arange(d) + 1, dyni=np.arange(d) + 1, difi=np.arange(d) + 1)
    Mt, St = mp.pred(dict(p=dict(w=g["W"], b=g["b"].T), maxU=g["e"]), plant,
                     dict(hyp=hyp_of(g["ell"], g["sf2"], g["sn2"]), inputs=g["X"], targets=g["Y"]), g["m"].T, g["s"], H)
    assert scaled_err(Mt, g["Mtraj"]) < 1e-12 and scaled_err(St, g["Straj"]) < 1e-11
    iK, beta = pp.calculate_factorizations(g["X"], g["Y"], g["ell"], g["sf2"], g["sn2"])
    Mp, Sp, _ = pp.predict(g["m"], g["s"], H, lambda m, s: pp.linear_action(g["W"], g["b"], m, s, True, g["e"]),
                           lambda m, s: pp.predict_given_factorizations(g["X"], g["ell"], g["sf2"], m, s, iK, beta),
                           lambda m, s: pp.exponential_reward(m, s, np.eye(d), np.zeros((1, d))))
    assert scaled_err(Mp[0], g["Mtraj"][:, -1]) < 1e-10 and scaled_err(Sp, g["Straj"][:, :, -1]) < 1e-9


def test_golden_regenerates_from_reference_sources():
    """Re-execute two of the reference's .m files (the checksummed copies under tests/reference_tests) with
    oracle/mrun.py and compare with the committed vectors."""
    from oracle import mrun
    g = load("gp0_a")
    M, S, V = mrun.run("gp0", dict(hyp=hyp_of(g["ell"], g["sf2"], g["sn2"]), inputs=g["X"], targets=g["Y"]), g["m"].T, g["s"], nout=3)
    # gp0.m goes through BLAS, whose summation order depends on the host's CPU kernel and thread count: over OpenBLAS
    # core types x 1-8 threads the vectors reproduce to <= 1.4e-14 (M), 2.7e-12 (S, cancellation), 2.7e-14 (V)
    assert scaled_err(M, g["M"]) < 1e-13 and scaled_err(S, g["S"]) < 1e-11 and scaled_err(V, g["V"]) < 1e-13
    g = load("gSin")
    M, S, C = mrun.run("gSin", g["m"].T, g["s"], float(g["e"]), nout=3)
    assert np.array_equal(M, g["M"]) and np.array_equal(S, g["S"])


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gp0_a", "gp0_b", "gp0_metric"])
def test_device_gp0_matches_golden(name):
    from pilco_b200 import engine
    g = load(name)
    gp = engine.gp_factorize(g["X"], g["Y"], g["ell"], g["sf2"], g["sn2"])
    M, S, V, info = engine.mm_forward(gp, g["m"], g["s"][None])
    assert int(info[0]) == 0
    assert scaled_err(M[0].cpu().numpy(), g["M"][:, 0]) < 1e-9
    assert scaled_err(S[0].cpu().numpy(), g["S"]) < 1e-7
    assert scaled_err(V[0].cpu().numpy(), g["V"]) < 1e-8


@pytest.mark.gpu
def test_device_gp1_gp2_match_golden():
    from pilco_b200 import engine
    g = load("gp1")
    gp = engine.fitc_factorize(g["X"], g["Z"], g["Y"], g["ell"], g["sf2"], g["sn2"])
    M, S, V, info = engine.mm_forward(gp, g["m"], g["s"][None])
    assert scaled_err(M[0].cpu().numpy(), g["M"][:, 0]) < 1e-6       # FITC: cond ~1e10 with the 1e-6 ridge
    assert scaled_err(S[0].cpu().numpy(), g["S"]) < 1e-5
    assert scaled_err(V[0].cpu().numpy(), g["V"]) < 1e-6
    g = load("gp2")
    gp = engine.gp_factorize(g["X"], g["Y"], g["ell"], np.ones(2), 1e-4 * np.ones(2), need_iK=False, mode=1)
    M, S, V, info = engine.mm_forward(gp, g["m"], g["s"][None])
    assert scaled_err(M[0].cpu().numpy(), g["M"][:, 0]) < 1e-7
    assert scaled_err(S[0].cpu().numpy(), g["S"]) < 1e-6
    assert scaled_err(V[0].cpu().numpy(), g["V"]) < 1e-7


@pytest.mark.gpu
def test_device_closed_forms_and_cascade_match_golden():
    from pilco_b200 import engine, _lib
    g = load("conlin")
    M, S, V = engine.linear_action(g["W"], g["b"][0], g["m"], g["s"][None])
    assert scaled_err(M[0].cpu().numpy(), g["M"][:, 0]) < 1e-14 and scaled_err(S[0].cpu().numpy(), g["S"]) < 1e-13
    g = load("gSin")
    M, S, C = engine.squash_sin(g["m"], g["s"][None], np.full(3, float(g["e"])))
    assert scaled_err(M[0].cpu().numpy(), g["M"][:, 0]) < 1e-13 and scaled_err(S[0].cpu().numpy(), g["S"]) < 1e-12
    assert scaled_err(C[0].cpu().numpy(), g["C"]) < 1e-13
    for k in (2, 5):
        g = load("reward_%d" % k)
        mu, sR = engine.exp_reward(g["W"], g["t"][0], g["m"], g["s"][None])
        assert abs(float(mu[0]) - g["muR"].item()) < 1e-13 and abs(float(sR[0]) - g["sR"].item()) < 1e-13
    g = load("pred")
    d = g["m"].shape[1]
    H = int(g["H"])
    gp = engine.gp_factorize(g["X"], g["Y"], g["ell"], g["sf2"], g["sn2"])
    spec = dict(kind=_lib.POLICY_LINEAR, Ds=d, U=1, squash=True, max_action=g["e"].ravel(), W=g["W"], b=g["b"][0])
    plan = engine.RolloutPlan(gp, spec, [dict(kind=_lib.REWARD_EXP, coef=1.0, W=np.eye(d), t=np.zeros(d))],
                              g["m"][0], g["s"], H, R=1)
    tm, tS, _ = plan.forward()
    # every step of the trajectory, not only the last one (test_cascade.py:74-78 checks the last at rtol 2e-4)
    assert scaled_err(tm[0].cpu().numpy().T, g["Mtraj"]) < 1e-8
    assert scaled_err(np.moveaxis(tS[0].cpu().numpy(), 0, -1), g["Straj"]) < 1e-7
