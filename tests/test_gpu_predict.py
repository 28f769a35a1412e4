"""pilco_gp_predict on the B200: GP predictive at deterministic test points (GPflow GPR / GPRFITC predict_f, predict_y,
predict_log_density on MGPR / SMGPR and their per-output models) against the numpy GPflow oracle, consistency with the
moment match at s = 0, bitwise reproducibility and the model-state paths (append, hyper-parameter change)."""
import numpy as np
import pytest
import torch

from gp_predict_oracle import predict_f as oracle_predict_f
from util import make_gp_problem

pytestmark = pytest.mark.gpu

BS = (1, 63, 65, 5000)


def _points(B, D, seed=5):
    return np.random.RandomState(seed).rand(B, D) * 1.2 - 0.1       # a margin outside the data's unit cube


def _check(mean, var, m0, v0, sf2, what=""):
    mean, var = np.asarray(mean), np.asarray(var)
    assert np.max(np.abs(mean - m0)) <= 1e-10 * np.max(np.abs(m0)), what
    assert np.max(np.abs(var - v0)) <= 1e-9 * np.max(sf2), what


@pytest.fixture(scope="module")
def engine():
    from pilco_b200 import engine
    return engine


@pytest.mark.parametrize("sn2", [1e-2, 1e-3])
@pytest.mark.parametrize("n,D,E", [(37, 3, 2), (300, 12, 10), (500, 10, 8), (600, 16, 3)])
def test_exact_gp_matches_gpflow_oracle(engine, n, D, E, sn2):
    X, Y, ell, sf2, _ = make_gp_problem(n, D, E, seed=n + D)
    sn = sn2 * np.ones(E)
    gp = engine.gp_factorize(X, Y, ell, sf2, sn)
    Xs = _points(max(BS), D)
    m0, v0 = oracle_predict_f(X, Y, ell, sf2, sn, Xs)
    for B in BS:
        mean, var = engine.gp_predict(gp, Xs[:B])
        assert mean.shape == (B, E) and var.shape == (B, E)
        _check(mean.cpu(), var.cpu(), m0[:B], v0[:B], sf2, "B=%d" % B)


@pytest.mark.parametrize("sn2", [1e-2, 1e-3])
def test_fitc_matches_gpflow_oracle(engine, sn2):
    """BASELINE sparse shape: N = 2000, M = 200 inducing points, E = 10, D = 12."""
    N, M, D, E = 2000, 200, 12, 10
    X, Y, ell, sf2, _ = make_gp_problem(N, D, E, seed=7)
    sn = sn2 * np.ones(E)
    Z = X[np.random.RandomState(8).choice(N, M, replace=False)] + 0.01
    gp = engine.fitc_factorize(X, Z, Y, ell, sf2, sn)
    Xs = _points(5000, D)
    m0, v0 = oracle_predict_f(X, Y, ell, sf2, sn, Xs, Z=Z)
    for B in BS:
        mean, var = engine.gp_predict(gp, Xs[:B])
        _check(mean.cpu(), var.cpu(), m0[:B], v0[:B], sf2, "B=%d" % B)


def test_full_cov(engine):
    n, D, E, B = 300, 12, 10, 200
    X, Y, ell, sf2, sn2 = make_gp_problem(n, D, E, seed=21)
    gp = engine.gp_factorize(X, Y, ell, sf2, sn2)
    Xs = _points(B, D, seed=22)
    mean, cov = engine.gp_predict(gp, Xs, full_cov=True)
    md, vd = engine.gp_predict(gp, Xs)
    mean, cov, md, vd = mean.cpu().numpy(), cov.cpu().numpy(), md.cpu().numpy(), vd.cpu().numpy()
    assert cov.shape == (E, B, B)
    assert np.array_equal(mean, md)
    s = np.max(sf2)
    assert np.max(np.abs(np.diagonal(cov, axis1=1, axis2=2).T - vd)) <= 1e-12 * s
    assert np.array_equal(cov, cov.transpose(0, 2, 1))
    m0, c0 = oracle_predict_f(X, Y, ell, sf2, sn2, Xs, full_cov=True)
    _check(mean, cov, m0, c0, sf2)
    Z = X[:60] + 0.01                                                     # FITC factors through the same path
    gpf = engine.fitc_factorize(X, Z, Y, ell, sf2, sn2)
    mf, cf = engine.gp_predict(gpf, Xs, full_cov=True)
    m0, c0 = oracle_predict_f(X, Y, ell, sf2, sn2, Xs, Z=Z, full_cov=True)
    _check(mf.cpu(), cf.cpu(), m0, c0, sf2)


def _mgpr(n=300, D=12, E=10, seed=31, sn2=1e-3, cls=None, **kw):
    from pilco_b200.models import MGPR
    X, Y, ell, sf2, _ = make_gp_problem(n, D, E, seed=seed)
    mg = (cls or MGPR)((X, Y), **kw)
    for e, m in enumerate(mg.models):
        m.kernel.lengthscales.assign(ell[e])
        m.kernel.variance.assign(sf2[e])
        m.likelihood.variance.assign(sn2)
    return mg


def _oracle_of(mg, Xs, Z=None):
    return oracle_predict_f(mg.X, mg.Y, mg.lengthscales, mg.variance, mg.noise, Xs, Z=Z)


def test_mgpr_predict_f_matches_moment_match_at_zero_input_variance():
    """predict_f(x) is the moment match at s = 0: M = mean, diag(S) = var, off-diagonal S = 0 (up to the cancellation of
    the E[f_a f_b] - M_a M_b terms)."""
    mg = _mgpr()
    Xs = _points(5, 12, seed=33)
    mean, var = mg.predict_f(Xs)
    D = Xs.shape[1]
    for b in range(5):
        M, S, _ = mg.predict_on_noisy_inputs(Xs[b:b + 1], np.zeros((D, D)))
        scale = max(np.max(mg.variance), np.max(M ** 2))
        assert np.max(np.abs(M[0] - mean[b])) <= 1e-10 * np.max(np.abs(M))
        assert np.max(np.abs(np.diag(S) - var[b])) <= 1e-9 * scale
        assert np.max(np.abs(S - np.diag(np.diag(S)))) <= 1e-9 * scale


def test_per_output_models_and_batch_position_are_bitwise():
    mg = _mgpr()
    Xs = _points(100000, 12, seed=41)
    mean, var = mg.predict_f(Xs)
    assert mean.shape == (100000, 10) and var.shape == (100000, 10)
    small = Xs[:700]
    m_all, v_all = mg.predict_f(small)
    for i, model in enumerate(mg.models):                                 # per-output model == column of the MGPR call
        mi, vi = model.predict_f(small)
        assert mi.shape == (700, 1) and vi.shape == (700, 1)
        assert np.array_equal(mi[:, 0], m_all[:, i]) and np.array_equal(vi[:, 0], v_all[:, i])
    for p in (0, 31, 32, 12345, 99999):                                   # alone == inside 1e5 points
        m1, v1 = mg.predict_f(Xs[p:p + 1])
        assert np.array_equal(m1[0], mean[p]) and np.array_equal(v1[0], var[p])
    mean2, var2 = mg.predict_f(Xs)                                        # two runs, same bits
    assert np.array_equal(mean, mean2) and np.array_equal(var, var2)
    m0, v0 = _oracle_of(mg, Xs[:2000])
    _check(mean[:2000], var[:2000], m0, v0, mg.variance)


def test_cuda_graph_replay_equals_eager(engine):
    mg = _mgpr()
    gp = mg.device_gp()
    Xs = engine.dev(_points(1000, 12, seed=51))
    me, ve = engine.gp_predict(gp, Xs)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        mg_, vg_ = engine.gp_predict(gp, Xs)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(me, mg_) and torch.equal(ve, vg_)
    Xs.copy_(engine.dev(_points(1000, 12, seed=52)))                    # replay with new points in the captured buffer
    g.replay()
    m2, v2 = engine.gp_predict(gp, Xs)
    torch.cuda.synchronize()
    assert torch.equal(m2, mg_) and torch.equal(v2, vg_)


def test_predictions_follow_append_and_hyperparameter_changes():
    """After an append the factors carry the block-inverse update's round-off, which grows with cond(K + sn2 I): that
    step is held to the bar the append path itself meets (1e-9 of the scale, test_gpu_forward.py), at sn2 = 1e-2 as
    there (at 1e-3 the appended factors are off by 1.3e-9).  A hyper-parameter change refactorises: the bars above."""
    mg = _mgpr(n=200, sn2=1e-2)
    Xs = _points(300, 12, seed=61)
    mg.predict_f(Xs)
    X1, Y1, _, _, _ = make_gp_problem(240, 12, 10, seed=62)
    mg.set_data((np.vstack([mg.X, X1[:40]]), np.vstack([mg.Y, Y1[:40]])))
    mean, var = mg.predict_f(Xs)
    assert mg.last_update == "append"
    m0, v0 = _oracle_of(mg, Xs)
    assert np.max(np.abs(mean - m0)) <= 1e-9 * np.max(np.abs(m0))
    assert np.max(np.abs(var - v0)) <= 1e-9 * np.max(mg.variance)
    mg.models[3].kernel.lengthscales.assign(1.3 * np.asarray(mg.models[3].kernel.lengthscales))
    mg.models[5].kernel.variance.assign(2.5)
    mean, var = mg.predict_f(Xs)
    assert mg.last_update == "factorize"
    m0, v0 = _oracle_of(mg, Xs)
    _check(mean, var, m0, v0, mg.variance, "assign")


def test_smgpr_predict_f_matches_fitc_oracle():
    """SMGPR predicts with the FITC factors its moment match uses: the inducing inputs of output 0 (smgpr.py:47-52)."""
    from pilco_b200.models import SMGPR
    mg = _mgpr(n=2000, seed=71, cls=SMGPR, num_induced_points=200)
    Z = mg.X[np.random.RandomState(72).choice(2000, 200, replace=False)] + 0.01
    mg.models[0].inducing_variable.Z.assign(Z)
    Xs = _points(3000, 12, seed=73)
    mean, var = mg.predict_f(Xs)
    m0, v0 = _oracle_of(mg, Xs, Z=np.asarray(mg.Z))
    _check(mean, var, m0, v0, mg.variance)
    mi, vi = mg.models[4].predict_f(Xs)
    assert np.array_equal(mi[:, 0], mean[:, 4]) and np.array_equal(vi[:, 0], var[:, 4])


def test_predict_y_and_log_density():
    from scipy.stats import norm
    mg = _mgpr()
    Xs = _points(500, 12, seed=81)
    Yt = np.random.RandomState(82).randn(500, 10) * 0.3
    mean, var = mg.predict_f(Xs)
    my, vy = mg.predict_y(Xs)
    assert np.array_equal(my, mean)
    assert np.max(np.abs(vy - (var + mg.noise))) <= 1e-15 * np.max(vy)
    ld = mg.predict_log_density((Xs, Yt))
    ref = norm.logpdf(Yt, loc=mean, scale=np.sqrt(var + mg.noise))
    assert ld.shape == (500, 10)
    assert np.max(np.abs(ld - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref)))
    m2 = mg.models[2]
    l2 = m2.predict_log_density((Xs, Yt[:, 2:3]))
    assert l2.shape == (500,) and np.array_equal(l2, ld[:, 2])
    y2, c2 = m2.predict_y(Xs[:50], full_cov=True)
    f2, cf2 = m2.predict_f(Xs[:50], full_cov=True)
    assert c2.shape == (1, 50, 50)
    assert np.array_equal(c2[0] - np.diag(np.diag(c2[0])), cf2[0] - np.diag(np.diag(cf2[0])))
    assert np.max(np.abs(np.diag(c2[0]) - np.diag(cf2[0]) - mg.noise[2])) <= 1e-15 * np.max(np.diag(c2[0]))


def test_notebook_one_step_prediction_loop():
    """examples/"Hyperparameter setting and troubleshooting tips.ipynb", "Check the one-step predictions manually"."""
    from pilco_b200.models import PILCO
    Ds, U, T = 4, 1, 40
    X, Y, ell, sf2, sn2 = make_gp_problem(150, Ds + U, Ds, seed=91)
    pilco = PILCO((X, Y), horizon=10)
    X_new = _points(T, Ds + U, seed=92)
    for i, m in enumerate(pilco.mgpr.models):
        y_pred_test, var_pred_test = m.predict_y(X_new)
        assert y_pred_test.shape == (T, 1) and var_pred_test.shape == (T, 1)
        assert np.all(np.isfinite(y_pred_test)) and np.all(var_pred_test > 0)
