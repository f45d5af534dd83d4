"""Joint_RF_SWD — mirror of /root/reference/model/model_rf_swd_vs_thk.py (:5-86).

`misfit_and_grad(x)` keeps the reference contract `(misfit, grad[2n], dsyn[ndata], flag)` with the
failure convention `(0.0, zeros, dobs, False)` (:73-74), and adds `misfit_and_grad_batch(X)` /
`device_context()` for the many-chains path (one fused CUDA evaluation for all rows of X).  The
parameterisation (`vpvs`, model/param.py) is the two sub-models' own: they must agree."""
import numpy as np
from .model_rf import ReceiverFunc
from .model_surf import SurfWD
from .._lib import Context
from . import param


class Joint_RF_SWD:
    def __init__(self, sigma1, sigma2, rfmodel: ReceiverFunc, swdmodel: SurfWD) -> None:
        if getattr(rfmodel, "vpvs", False) != getattr(swdmodel, "vpvs", False):
            raise ValueError(f"the receiver-function model has vpvs={rfmodel.vpvs} and the dispersion model "
                             f"vpvs={swdmodel.vpvs}: a joint model needs one parameterisation")
        self.sigma1 = sigma1
        self.sigma2 = sigma2
        self.rfmodel = rfmodel
        self.swdmodel = swdmodel
        self.ndata = rfmodel.nt + swdmodel.nt
        self.which = 0
        self._ctx = None
        self._ctx_key = None
        self._device = 0

    @property
    def vpvs(self):
        return self.rfmodel.vpvs

    @property
    def npar(self):
        return param.npar(self.vpvs)

    def set_obsdata(self, rfobs: np.ndarray, swdobs: np.ndarray):
        self.dobs = np.zeros((self.ndata))
        self.rfobs = rfobs * 1.
        self.swdobs = swdobs * 1.
        self.rfmodel.set_obsdata(rfobs)
        self.swdmodel.set_obsdata(swdobs)
        self.dobs[:self.rfmodel.nt] = self.rfobs * 1.
        self.dobs[self.rfmodel.nt:] = self.swdobs * 1.

    def set_device(self, device):
        """GPU of this model and of its two sub-models."""
        self.rfmodel.set_device(device)
        self.swdmodel.set_device(device)
        if device != self._device:
            self._device = device
            self._ctx = None
            self._ctx_key = None

    def device_context(self, n):
        """Configured rfs context (joint model + observations) for n layers.  The configuration is
        re-pushed whenever a field the reference reads per call has changed (sigma1/2, every field of
        the two sub-models, the observations): model_rf_swd_vs_thk.py:66-86."""
        if self._ctx is None:
            self._ctx = Context(self._device)
        key = (self.sigma1, self.sigma2) + self._config_fields(n) + (
            np.asarray(self.dobs, dtype=np.float64).tobytes(),)
        if self._ctx_key != key:
            self._config_forward(self._ctx, n)
            self._ctx.config_obs(self.dobs, self.sigma1, self.sigma2)
            self._ctx_key = key
        return self._ctx

    def _config_fields(self, n):
        return (self.rfmodel._config_fields(n), self.swdmodel._config_fields(n))

    def _config_forward(self, ctx, n):
        self.swdmodel._config_forward(ctx, n)
        self.rfmodel._config_forward(ctx, n)

    def forward(self, x: np.ndarray):
        drf = self.rfmodel.forward(x)
        dswd, flag = self.swdmodel.forward(x)
        return drf, dswd, flag

    def misfit(self, x: np.ndarray):
        drf, dswd, flag = self.forward(x)
        if flag:
            n1 = drf.size
            n2 = dswd.size
            wt = (self.sigma1 / self.sigma2)**2 * n1 / n2
            misfit = 0.5 * np.sum((drf - self.rfobs)**2) + 0.5 * np.sum((dswd - self.swdobs)**2) * wt
            return misfit, True
        return 0.0, flag

    def misfit_and_grad_batch(self, X):
        """X [B, P n] -> (U[B], grad[B,P n], dsyn[B,ndata], flag[B]) in one fused GPU evaluation."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        return self.device_context(param.layer_count(X.shape[1], self.vpvs)).misfit_grad_host(X, which=0)

    def misfit_and_grad(self, x: np.ndarray):
        x = np.asarray(x, dtype=np.float64)
        U, g, d, f = self.misfit_and_grad_batch(x[None, :])
        if not f[0]:
            return 0.0, np.zeros(x.shape), self.dobs, False
        return float(U[0]), g[0], d[0], True
