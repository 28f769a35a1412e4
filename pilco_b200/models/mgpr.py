"""MGPR -- E independent SE-ARD GPs sharing their inputs, predicted at a Gaussian input by moment
matching on the device (drop-in for the reference class at pilco/models/mgpr.py:17-190).

Host side (this file): parameter objects, data handling, training driver.
Device side: ``pilco_gp_factorize`` (mgpr.py:81-89) and ``pilco_mm_forward`` (mgpr.py:91-149) through
``pilco_b200.engine``.  Factorisations are cached per (data, hyper-parameter) state instead of being
recomputed on every call as the reference does (mgpr.py:77-79).
"""
import numpy as np
import torch

from .. import engine, gp_training
from ..params import Parameter, Softplus, host


class Kernel:
    """SE-ARD kernel parameter holder (gpflow.kernels.SquaredExponential surface)."""

    def __init__(self, D, lengthscale_lower=0.0):
        self.lengthscales = Parameter(np.ones(D), transform=Softplus(lengthscale_lower), name="lengthscales")
        self.variance = Parameter(1.0, transform=Softplus(0.0), name="variance")

    def K(self, X1, X2=None):
        X1 = np.asarray(X1, dtype=np.float64)
        X2 = X1 if X2 is None else np.asarray(X2, dtype=np.float64)
        ell = np.asarray(self.lengthscales)
        a, b = X1 / ell, X2 / ell
        d2 = (a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * a @ b.T
        return float(self.variance) * np.exp(-0.5 * np.maximum(d2, 0.0))


class Likelihood:
    def __init__(self, variance=1.0):
        self.variance = Parameter(variance, transform=Softplus(1e-6), name="likelihood_variance")
        self.prior = None


class GPRModel:
    """One output GP: kernel + Gaussian likelihood + its (X, y) data (gpflow.models.GPR surface)."""

    def __init__(self, data, kernel):
        self.data = (np.asarray(data[0], dtype=np.float64), np.asarray(data[1], dtype=np.float64))
        self.kernel = kernel
        self.likelihood = Likelihood(1.0)

    @property
    def parameters(self):
        return [self.kernel.lengthscales, self.kernel.variance, self.likelihood.variance]

    @property
    def trainable_parameters(self):
        return [p for p in self.parameters if p.trainable]

    def _loss(self, vals):
        X = torch.as_tensor(np.asarray(self.data[0]), dtype=torch.float64)
        y = torch.as_tensor(np.asarray(self.data[1]), dtype=torch.float64)[:, 0]
        ell, sf2, sn2 = vals
        return gp_training.gpr_loss(X, y, ell, sf2, sn2,
                                    ell_prior=self.kernel.lengthscales.prior, sf2_prior=self.kernel.variance.prior)

    def training_loss(self):
        return float(self._loss([torch.as_tensor(p.value(), dtype=torch.float64) for p in self.parameters]))

    def optimize(self, maxiter=None):
        return gp_training.minimize(self._loss, self.parameters, maxiter=maxiter)

    # ---- gpflow prediction surface: routed through the owning MGPR / SMGPR (its resident device model, output i) -----
    def _owner(self):
        owner = getattr(self, "_mgpr", None)
        if owner is None:
            raise RuntimeError("GPRModel predictions run on the device model of the MGPR / SMGPR that created it")
        return owner, self._output

    def predict_f(self, Xnew, full_cov=False):
        """gpflow GPR.predict_f: latent mean [B,1] and variance [B,1] (or covariance [1,B,B] with ``full_cov``)."""
        owner, i = self._owner()
        return owner._predict(Xnew, full_cov, output=i)

    def predict_y(self, Xnew, full_cov=False):
        """gpflow GPR.predict_y: predict_f plus the likelihood variance."""
        owner, i = self._owner()
        return owner._predict(Xnew, full_cov, output=i, noise=True)

    def predict_log_density(self, data):
        """gpflow GPR.predict_log_density: log N(y | mean, var + sn2) per point, [B]."""
        owner, i = self._owner()
        return owner._log_density(data, output=i)[:, 0]


def randomize(model, mean=1, sigma=0.01):
    """pilco/models/mgpr.py:8-15"""
    model.kernel.lengthscales.assign(mean + sigma * np.random.normal(size=model.kernel.lengthscales.shape))
    model.kernel.variance.assign(mean + sigma * np.random.normal(size=model.kernel.variance.shape))
    if model.likelihood.variance.trainable:
        model.likelihood.variance.assign(mean + sigma * np.random.normal())


class MGPR:
    mm_mode = 0         # 0: GP with trace term; 1: deterministic GP (RbfController)

    def __init__(self, data, name=None):
        self.name = name
        self.num_outputs = data[1].shape[1]
        self.num_dims = data[0].shape[1]
        self.num_datapoints = data[0].shape[0]
        self.create_models(data)
        self.optimizers = []
        self._cache_key = None
        self._cache_gp = None

    # ---- construction / data (mgpr.py:28-45) -------------------------------------------------
    def create_models(self, data):
        self.models = []
        for i in range(self.num_outputs):
            kern = Kernel(data[0].shape[1])
            kern.lengthscales.prior = (1.1, 1.0 / 10.0)        # Gamma(alpha, rate)   mgpr.py:33
            kern.variance.prior = (1.5, 1.0 / 2.0)             # mgpr.py:34
            self.models.append(GPRModel((data[0], data[1][:, i:i + 1]), kern))
        self._own_models()

    def _own_models(self):
        """Back-reference from each per-output model to this MGPR: its gpflow prediction methods run here."""
        for i, model in enumerate(self.models):
            model._mgpr, model._output = self, i

    def set_data(self, data):
        for i, model in enumerate(self.models):
            if isinstance(model.data[0], Parameter):
                model.X.assign(data[0])
                model.Y.assign(data[1][:, i:i + 1])
                model.data = [model.X, model.Y]
            else:
                model.data = (np.asarray(data[0], dtype=np.float64), np.asarray(data[1][:, i:i + 1], dtype=np.float64))
        self.num_datapoints = np.asarray(data[0]).shape[0]

    # ---- training (mgpr.py:47-75) -----------------------------------------------------------------
    def optimize(self, restarts=1, maxiter=None):
        """All outputs and restarts in lock step on the device (pilco_gp_nlml; gp_device_training.py)."""
        from .. import gp_device_training
        self.optimizers = [True] * len(self.models)
        return gp_device_training.optimize_mgpr(self, restarts=restarts, maxiter=maxiter)

    def optimize_host(self, restarts=1, maxiter=None):
        """Host path (torch-CPU autograd + SciPy): used by SMGPR (FITC objective, gp_training.py)."""
        for model in self.models:
            model.optimize(maxiter)
        self.optimizers = [True] * len(self.models)
        for model in self.models:
            best = [p.value() for p in model.parameters]
            best_loss = model.training_loss()
            for _ in range(restarts):
                randomize(model)
                model.optimize(maxiter)
                loss = model.training_loss()
                if loss < best_loss:          # the reference's bookkeeping keeps the last restart
                    best_loss = loss          # (mgpr.py:58-75); keeping the best is the documented intent
                    best = [p.value() for p in model.parameters]
            for p, v in zip(model.parameters, best):
                p.assign(v)

    @property
    def trainable_parameters(self):
        return [p for m in self.models for p in m.trainable_parameters]

    @property
    def parameters(self):
        return [p for m in self.models for p in m.parameters]

    # ---- stacked views (mgpr.py:151-190) -------------------------------------------------------
    @property
    def X(self):
        return np.asarray(self.models[0].data[0], dtype=np.float64)

    @property
    def Y(self):
        return np.concatenate([np.asarray(m.data[1], dtype=np.float64) for m in self.models], axis=1)

    @property
    def data(self):
        return (self.X, self.Y)

    @property
    def lengthscales(self):
        return np.stack([np.asarray(m.kernel.lengthscales) for m in self.models])

    @property
    def variance(self):
        return np.stack([np.asarray(m.kernel.variance) for m in self.models]).reshape(-1)

    @property
    def noise(self):
        return np.stack([np.asarray(m.likelihood.variance) for m in self.models]).reshape(-1)

    def centralized_input(self, m):
        return self.centres - np.asarray(m)

    @property
    def centres(self):
        return self.X

    def K(self, X1, X2=None):
        return np.stack([m.kernel.K(X1, X2) for m in self.models])

    # ---- device path ---------------------------------------------------------------------------
    def _state_key(self):
        parts = [self.X, self.Y, self.lengthscales, self.variance, self.noise]
        return hash(tuple(np.ascontiguousarray(p).tobytes() for p in parts))

    def _factorize(self):
        return engine.gp_factorize(self.X, self.Y, self.lengthscales, self.variance, self.noise,
                                   need_iK=(self.mm_mode == 0), mode=self.mm_mode)

    # incremental set_data (SURVEY section 8f-2): rows appended + hyper-parameters unchanged -> O(n^2 k) update of the
    # resident inverse instead of a new O(n^3) factorisation.  After MAX_APPENDS consecutive appends (round-off of
    # the block-inverse recursion) or when more rows arrive than the model holds, it is refactorised from scratch.
    MAX_APPENDS = 8
    incremental = True

    def _hyper_key(self):
        return hash(tuple(np.ascontiguousarray(p).tobytes() for p in (self.lengthscales, self.variance, self.noise)))

    def _try_append(self):
        """The cached model extended by the appended rows, or None when this is not a pure append."""
        gp, snap = self._cache_gp, getattr(self, "_cache_snap", None)
        if not self.incremental or gp is None or snap is None or type(self)._factorize is not MGPR._factorize:
            return None
        X, Y = self.X, self.Y
        X0, Y0, hk = snap
        n0, n1 = X0.shape[0], X.shape[0]
        if not (n0 < n1 <= 2 * n0) or X.shape[1] != X0.shape[1] or Y.shape[1] != Y0.shape[1] or hk != self._hyper_key():
            return None
        if getattr(gp, "appends", 0) >= self.MAX_APPENDS:
            return None
        if not (np.array_equal(X[:n0], X0) and np.array_equal(Y[:n0], Y0)):
            return None
        new = engine.gp_append(gp, X, Y)
        return new if int(new.info.max().item()) == 0 else None

    def device_gp(self):
        """Factorised device model, resident until data or hyper-parameters change; appended rows update it in
        place of a refactorisation (``_try_append``)."""
        key = self._state_key()
        if key != self._cache_key:
            gp = self._try_append() if self.mm_mode == 0 else None
            self.last_update = "append" if gp is not None else "factorize"
            if gp is None:
                gp = self._factorize()
                bad = int(gp.info.max().item())
                if bad:
                    raise RuntimeError("Cholesky decomposition was not successful (Gram matrix not positive definite)")
            self._cache_gp, self._cache_key = gp, key
            self._cache_snap = (self.X.copy(), self.Y.copy(), self._hyper_key())
        return self._cache_gp

    def calculate_factorizations(self):
        """(iK [E,n,n], beta [E,n]) as CUDA tensors  (mgpr.py:81-89)."""
        gp = self.device_gp()
        iK = gp.iK[:, :gp.n, :gp.n] if gp.iK is not None else None
        self._last_fact = (iK, gp.beta, self._cache_key)
        return iK, gp.beta

    def _gp_from_factors(self, iK, beta):
        """Temporary device model around caller-supplied factors (any array-like [E,n,n] / [E,n]): the reference's
        predict_given_factorizations computes with whatever it is handed (mgpr.py:91-149; RbfController passes
        ``0.0 * iK``, controllers.py:116), so custom / modified factors must drive the result here too."""
        base = self.device_gp()
        n, E = base.n, base.E
        beta_d = engine.dev(beta.detach() if isinstance(beta, torch.Tensor) else beta).reshape(E, n)
        iK_d = engine.dev(iK.detach() if isinstance(iK, torch.Tensor) else iK).reshape(E, n, n)
        ldk = engine.pad_n(n)
        pad = torch.zeros((E, ldk, ldk), dtype=torch.float64, device=iK_d.device)
        pad[:, :n, :n] = iK_d
        return engine.DeviceGP(base.X, base.ell, base.sf2, beta_d, pad, ldk, mode=0)

    def predict_given_factorizations(self, m, s, iK=None, beta=None):
        """mgpr.py:91-149 on the device.  With no factors, or with exactly the objects ``calculate_factorizations``
        returned for the current state, the cached device model is used; any other ``iK`` / ``beta`` is honoured
        (a temporary device model is built from them) -- never silently ignored."""
        gp = self.device_gp()
        last = getattr(self, "_last_fact", None)
        own = last is not None and last[2] == self._cache_key and iK is last[0] and beta is last[1]
        if (iK is None) != (beta is None):
            raise ValueError("predict_given_factorizations: pass both iK and beta (or neither)")
        if iK is not None and not own:
            gp = self._gp_from_factors(iK, beta)
        m = np.asarray(m, dtype=np.float64).reshape(1, -1)
        s = np.asarray(s, dtype=np.float64).reshape(1, gp.D, gp.D)
        M, S, V, info = engine.mm_forward(gp, m, s)
        if int(info[0].item()):
            raise RuntimeError("moment matching failed: input covariance system not positive definite")
        return host(M), host(S[0]), host(V[0])

    def predict_on_noisy_inputs(self, m, s):
        """mgpr.py:77-79 -> (M [1,E], S [E,E], V [D,E])"""
        return self.predict_given_factorizations(m, s)

    # ---- prediction at deterministic inputs (gpflow GPR / GPRFITC.predict_f of every output at once) -------------------
    def _predict_device(self, Xnew, full_cov=False, output=None, noise=False):
        """pilco_gp_predict on the resident device model (``device_gp``: same cache, refactorisation and incremental
        append as the moment match).  CUDA tensors: mean [B,E'] and var [B,E'] or cov [E',B,B] (E' = 1 for ``output``)."""
        if self.mm_mode != 0:
            raise TypeError("%s is a deterministic GP (no predictive variance)" % type(self).__name__)
        gp = self.device_gp()
        sn2 = engine.dev(self.noise)
        if output is not None:
            gp, sn2 = gp.output(output), sn2[output:output + 1]
        X = np.asarray(Xnew, dtype=np.float64).reshape(-1, gp.D)
        mean, v = engine.gp_predict(gp, X, full_cov=full_cov)
        if noise:
            v = v + (torch.diag_embed(sn2[:, None].expand(-1, v.shape[-1])) if full_cov else sn2)
        return mean, v

    def _predict(self, Xnew, full_cov=False, output=None, noise=False):
        mean, v = self._predict_device(Xnew, full_cov, output, noise)
        return host(mean), host(v)

    def _log_density(self, data, output=None):
        mean, var = self._predict_device(data[0], output=output, noise=True)
        Y = engine.dev(np.asarray(data[1], dtype=np.float64).reshape(mean.shape))
        return host(-0.5 * (np.log(2.0 * np.pi) + torch.log(var) + (Y - mean) ** 2 / var))

    def predict_f(self, Xnew, full_cov=False):
        """Latent predictive of all E outputs at the points Xnew [B,D] (gpflow GPR.predict_f, or GPRFITC.predict_f under
        SMGPR): mean [B,E] and var [B,E], or cov [E,B,B] with ``full_cov``.  One device call."""
        return self._predict(Xnew, full_cov)

    def predict_y(self, Xnew, full_cov=False):
        """predict_f plus the likelihood variances ``noise`` (on the diagonal with ``full_cov``)."""
        return self._predict(Xnew, full_cov, noise=True)

    def predict_log_density(self, data):
        """Gaussian log density of Y [B,E] under predict_y at X [B,D], data = (X, Y): [B,E]."""
        return self._log_density(data)
