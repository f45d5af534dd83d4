"""ReceiverFunc — mirror of /root/reference/model/model_rf.py (class ReceiverFunc :4-197).

Same constructor / `init(**kargs)` / `set_obsdata` / `set_thk` / `empirical_relation` / `forward` /
`misfit` / `misfit_and_grad` (3-tuple, no flag, as the reference).  `misfit_and_grad` runs the fused
CUDA path (rfs_misfit_grad_host, which=1): propagator + spectral deconvolution + adjoint gradient.

Extensions: `ray_p` may be a list of ray parameters and `gauss` a list of Gaussian widths; the data
vector is then the concatenation of one trace per (ray parameter, width) in the order [ray][gauss]
(`nt` counts all of them, `nt_trace` one trace) and misfit / gradient sum over them — one objective per
chain instead of one model object per ray parameter and width.  With `vpvs=True` the model vector is
[vs, thk, vpvs] (model/param.py): each layer's Vp/Vs ratio is sampled instead of following Brocher's curve."""
import numpy as np
from .lib import librf
from .._lib import Context
from . import param


class ReceiverFunc:
    def __init__(self, ray_p, nt, dt, gauss, time_shift, water_level=0.001, type_="p", method="time", *,
                 vpvs=False):
        self.vpvs = bool(vpvs)
        self.ray_p = ray_p
        self.nray = int(np.size(ray_p))
        self.ngauss = int(np.size(gauss))
        self.nt_trace = nt
        # data count (== nt for the reference's single ray parameter and width)
        self.nt = nt * self.nray * self.ngauss
        self.dt = dt
        self.gauss = gauss
        self.time_shift = time_shift
        self.water_level = water_level
        self.rf_type = type_
        self.t = np.arange(nt) * dt - time_shift
        self.method = method
        self.which = 1
        self._ctx = None
        self._ctx_key = None
        self._device = 0

    @classmethod
    def init(self, **kargs):
        return ReceiverFunc(kargs['ray_p'], kargs['nt'], kargs['dt'], kargs['gauss'], kargs['time_shift'],
                            kargs['water_level'], kargs['type'], kargs['method'], vpvs=kargs.get('vpvs', False))

    def set_obsdata(self, dobs):
        self.dobs = dobs

    def set_device(self, device):
        if device != self._device:
            self._device = device
            self._ctx = None
            self._ctx_key = None

    def set_thk(self, thk):
        self.thk = thk * 1.0

    @property
    def npar(self):
        return param.npar(self.vpvs)

    def empirical_relation(self, vs, deriv=False, k=None):
        """Brocher vp and rho of vs; with k (Vp/Vs per layer) vp = k vs and dadb = k."""
        if k is not None:
            return param.brocher(vs, k, deriv)
        vp = 0.9409 + 2.0947 * vs - 0.8206 * vs**2 + 0.2683 * vs**3 - 0.0251 * vs**4
        rho = 1.6612 * vp - 0.4721 * vp**2 + 0.0671 * vp**3 - 0.0043 * vp**4 + 0.000106 * vp**5
        if deriv:
            drda = 1.6612 - 0.4721 * 2 * vp + 0.0671 * 3 * vp**2 - 0.0043 * 4 * vp**3 + 0.000106 * 5 * vp**4
            dadb = 2.0947 - 0.8206 * 2 * vs + 0.2683 * 3 * vs**2 - 0.0251 * 4 * vs**3
            return vp, rho, drda, dadb
        return vp, rho

    def _config_fields(self, n):
        # every field the reference reads on each misfit_and_grad call (model_rf.py:137-197): changing
        # one of them after the first call re-configures the device context
        gauss = self.gauss if np.ndim(self.gauss) == 0 else tuple(np.asarray(self.gauss, dtype=np.float64).tolist())
        return (n, tuple(np.atleast_1d(self.ray_p).tolist()), self.nt_trace, self.dt, gauss,
                self.time_shift, self.water_level, self.rf_type, self.method, self.vpvs)

    def _config_key(self, n):
        return self._config_fields(n) + (np.asarray(self.dobs, dtype=np.float64).tobytes(),)

    def device_context(self, n):
        """Configured rfs context (RF objective + observations) for n layers."""
        if self._ctx is None:
            self._ctx = Context(self._device)
        key = self._config_key(n)
        if self._ctx_key != key:
            self._config_forward(self._ctx, n)
            self._ctx.config_obs(self.dobs)
            self._ctx_key = key
        return self._ctx

    def _config_forward(self, ctx, n):
        ctx.config_param(self.vpvs)
        ctx.config_rf(n, self.ray_p, self.nt_trace, self.dt, self.gauss, self.time_shift, self.water_level,
                      self.rf_type, self.method)

    _context = device_context

    def forward(self, x: np.ndarray):
        if self.vpvs:
            vs, thk, k = param.split(x, True)
            vp, rho = self.empirical_relation(vs, k=k)
        else:
            layers = int(len(x) / 2)
            vs = x[:layers]
            thk = x[layers:]
            vp, rho = self.empirical_relation(vs, deriv=False)
        qa = thk * 0 + 9999.
        qb = thk * 0 + 9999.
        out = [librf.forward(thk, rho, vp, vs, qa, qb, float(p), self.nt_trace, self.dt, float(g),
                             self.time_shift, self.method, self.water_level, self.rf_type)
               for p in np.atleast_1d(self.ray_p) for g in np.atleast_1d(self.gauss)]
        return out[0] if len(out) == 1 else np.hstack(out)

    def misfit(self, x):
        d = self.forward(x)
        return 0.5 * np.sum((d - self.dobs)**2)

    def misfit_and_grad(self, x):
        x = np.asarray(x, dtype=np.float64)
        n = param.layer_count(x.shape[0], self.vpvs)
        U, g, d, _ = self.device_context(n).misfit_grad_host(x[None, :], which=1)
        return float(U[0]), g[0], d[0]

    def misfit_and_grad_batch(self, X):
        """X [B, P n] -> (U[B], grad[B,P n], dsyn[B,nt], flag[B]) in one fused GPU evaluation."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        return self.device_context(param.layer_count(X.shape[1], self.vpvs)).misfit_grad_host(X, which=1)
