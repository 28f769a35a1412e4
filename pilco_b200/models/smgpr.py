"""SMGPR -- FITC sparse variant (drop-in for pilco/models/smgpr.py:11-52).  The FITC factorisation
(smgpr.py:24-45, gp1.m:52-82) runs on the device (``pilco_fitc_factorize``); the moment match then runs
over the M inducing points of output 0 (smgpr.py:47-52).  ``predict_f`` / ``predict_y`` / ``predict_log_density``
(inherited from MGPR, and on every GPRFITCModel) use the same FITC factors, hence the inducing inputs of output 0 for
every output: GPRFITC.predict_f of each output when the outputs share their inducing inputs."""
import numpy as np
import torch

from .. import engine, gp_training
from ..params import Parameter
from .mgpr import MGPR, GPRModel, Kernel


class InducingPoints:
    def __init__(self, Z):
        self.Z = Parameter(Z, name="Z")


class GPRFITCModel(GPRModel):
    """gpflow.models.GPRFITC surface: adds trainable inducing inputs."""

    def __init__(self, data, kernel, inducing_variable):
        super().__init__(data, kernel)
        self.inducing_variable = InducingPoints(inducing_variable)

    @property
    def parameters(self):
        return [self.kernel.lengthscales, self.kernel.variance, self.likelihood.variance, self.inducing_variable.Z]

    def _loss(self, vals):
        X = torch.as_tensor(np.asarray(self.data[0]), dtype=torch.float64)
        y = torch.as_tensor(np.asarray(self.data[1]), dtype=torch.float64)[:, 0]
        ell, sf2, sn2, Z = vals
        return gp_training.fitc_loss(X, y, Z, ell, sf2, sn2)


class SMGPR(MGPR):
    def __init__(self, data, num_induced_points, name=None):
        self.num_induced_points = num_induced_points
        MGPR.__init__(self, data, name)

    def create_models(self, data):
        self.models = []
        for i in range(self.num_outputs):
            kern = Kernel(data[0].shape[1])
            Z = np.random.rand(self.num_induced_points, self.num_dims)      # smgpr.py:20
            self.models.append(GPRFITCModel((data[0], data[1][:, i:i + 1]), kern, Z))
        self._own_models()

    def optimize(self, restarts=1, maxiter=None):
        """FITC objective with trainable inducing inputs, on the device: all outputs and restarts in lock step, value
        and analytic gradient from ``pilco_fitc_nlml`` (gp_device_training.optimize_smgpr).  ``optimize_host`` keeps
        the torch-CPU autograd path as the cross-check the tests use."""
        from .. import gp_device_training
        self.optimizers = [True] * len(self.models)
        return gp_device_training.optimize_smgpr(self, restarts=restarts, maxiter=maxiter)

    @property
    def Z(self):
        return self.models[0].inducing_variable.Z                           # smgpr.py:50-52

    @property
    def centres(self):
        return np.asarray(self.Z)

    def _state_key(self):
        parts = [self.X, self.Y, self.lengthscales, self.variance, self.noise, np.asarray(self.Z)]
        return hash(tuple(np.ascontiguousarray(p).tobytes() for p in parts))

    def _factorize(self):
        return engine.fitc_factorize(self.X, np.asarray(self.Z), self.Y, self.lengthscales, self.variance, self.noise)
