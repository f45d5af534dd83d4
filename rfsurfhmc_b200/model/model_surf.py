"""SurfWD — mirror of /root/reference/model/model_surf.py (class SurfWD :4-228).

Same constructor, `init(**kargs)`, `set_obsdata`, `set_thk`, `empirical_relation`, `forward`,
`misfit`, `misfit_and_grad` and return shapes.  `misfit_and_grad` runs the fused CUDA path
(rfs_misfit_grad_host, which=2) instead of per-wave-type pybind calls + NumPy glue; `forward`
goes through the libsurf drop-in.  Reference quirks kept: Lc/Lg are evaluated on `tRc`
(model_surf.py:200-201,211-212) and `forward` evaluates Rg/Lc/Lg on `tRc` (:114-130); on a failed
root search the gradient has length n, not 2n (:179-180).

Extension: `mode` may be an ascending list of modes; the data vector is then [mode][Rc,Rg,Lc,Lg]
(`nt` counts all of them) and all modes come out of ONE chained root-search pass.  With `vpvs=True` the model vector is
[vs, thk, vpvs] (model/param.py): each layer's Vp/Vs ratio is sampled instead of following Brocher's curve."""
import numpy as np
from .lib import libsurf
from .._lib import Context
from . import param


class SurfWD:
    def __init__(self, mode=0, sphere=False, tRc=None, tRg=None, tLc=None, tLg=None, *, vpvs=False):
        self.vpvs = bool(vpvs)
        self.mode = mode
        self.nmode = int(np.size(mode))
        self.sphere = sphere
        self.which = 2
        self._device = 0
        self.tRc, self.tRg, self.tLc, self.tLg = None, None, None, None
        self.nt = 0
        self.ntRc, self.ntRg, self.ntLc, self.ntLg = 0, 0, 0, 0
        if tRc is not None and len(tRc) > 0:
            self.tRc = np.asarray(tRc)
            self.ntRc = len(tRc)
            self.nt += self.ntRc
        if tRg is not None and len(tRg) > 0:
            self.tRg = np.asarray(tRg)
            self.ntRg = len(tRg)
            self.nt += self.ntRg
        if tLc is not None and len(tLc) > 0:
            self.tLc = np.asarray(tLc)
            self.ntLc = len(tLc)
            self.nt += self.ntLc
        if tLg is not None and len(tLg) > 0:
            self.tLg = np.asarray(tLg)
            self.ntLg = len(tLg)
            self.nt += self.ntLg
        self.nt *= self.nmode
        self._ctx = None
        self._ctx_key = None

    @classmethod
    def init(self, **kargs):
        return SurfWD(tRc=kargs['tRc'], tRg=kargs['tRg'], tLc=kargs['tLc'], tLg=kargs['tLg'],
                      vpvs=kargs.get('vpvs', False))

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

    def empirical_relation(self, vs: np.ndarray, deriv=False, k=None):
        """Brocher vp and rho of vs (and dadb, drda); with k (Vp/Vs per layer) vp = k vs and dadb = k."""
        if k is not None:
            vp, rho, drda, dadb = param.brocher(vs, k, True)
            return (vp, rho, dadb, drda) if deriv else (vp, rho)
        vp = 0.9409 + 2.0947 * vs - 0.8206 * vs**2 + 0.2683 * vs**3 - 0.0251 * vs**4
        rho = 1.6612 * vp - 0.4721 * vp**2 + 0.0671 * vp**3 - 0.0043 * vp**4 + 0.000106 * vp**5
        dadb = np.zeros(vp.shape)
        drda = np.zeros((vp.shape))
        if deriv:
            drda = 1.6612 - 0.4721 * 2 * vp + 0.0671 * 3 * vp**2 - 0.0043 * 4 * vp**3 + 0.000106 * 5 * vp**4
            dadb = 2.0947 - 0.8206 * 2 * vs + 0.2683 * 3 * vs**2 - 0.0251 * 4 * vs**3
        if deriv is False:
            return vp, rho
        return vp, rho, dadb, drda

    # period lists as the reference's misfit_and_grad passes them (quirk: Love uses tRc)
    def _grad_periods(self):
        lc = self.tRc[:self.ntLc] if self.ntLc > 0 else None
        lg = self.tRc[:self.ntLg] if self.ntLg > 0 else None
        if (self.ntLc > 0 and self.ntLc != self.ntRc) or (self.ntLg > 0 and self.ntLg != self.ntRc):
            raise ValueError("reference quirk: Lc/Lg are evaluated on tRc, so len(tLc)/len(tLg) must "
                             "equal len(tRc) (model/model_surf.py:200-201,211-212)")
        return self.tRc, self.tRg, lc, lg

    def _config_fields(self, n):
        # every field the reference reads on each misfit_and_grad call (model_surf.py:155-228)
        per = tuple(None if t is None else np.asarray(t, dtype=np.float64).tobytes()
                    for t in self._grad_periods())
        return (n, tuple(np.atleast_1d(self.mode).tolist()), bool(self.sphere), per, self.vpvs)

    def _config_key(self, n):
        return self._config_fields(n) + (np.asarray(self.dobs, dtype=np.float64).tobytes(),)

    def device_context(self, n):
        """Configured rfs context (SWD objective + observations) for n layers."""
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
        tRc, tRg, tLc, tLg = self._grad_periods()
        ctx.config_swd(n, tRc, tRg, tLc, tLg, mode=self.mode, sphere=self.sphere)

    _context = device_context

    def forward(self, x: np.ndarray):
        d = np.zeros((self.nt))
        if self.vpvs:
            vs, thk, k = param.split(x, True)
            vp, rho = self.empirical_relation(vs, k=k)
        else:
            layers = int(len(x) / 2)
            vs = x[:layers]
            thk = x[layers:]
            vp, rho = self.empirical_relation(vs)
        k1 = 0
        for mode in np.atleast_1d(self.mode):
            for nt_w, wt in ((self.ntRc, "Rc"), (self.ntRg, "Rg"), (self.ntLc, "Lc"), (self.ntLg, "Lg")):
                if nt_w > 0:
                    k2 = k1 + nt_w
                    d[k1:k2], flag = libsurf.forward(thk, vp, vs, rho, self.tRc, wt, int(mode), self.sphere)
                    if flag is False:
                        return d, flag
                    k1 = k2
        return d, True

    def misfit(self, x):
        d, flag = self.forward(x)
        if flag:
            return 0.5 * np.sum((d - self.dobs)**2), True
        return 0.0, flag

    def misfit_and_grad(self, x):
        x = np.asarray(x, dtype=np.float64)
        n = param.layer_count(x.shape[0], self.vpvs)
        U, g, d, f = self.device_context(n).misfit_grad_host(x[None, :], which=2)
        if not f[0]:
            return 0.0, np.zeros((n)), d[0], False
        return float(U[0]), g[0], d[0], True

    def misfit_and_grad_batch(self, X):
        """X [B, P n] -> (U[B], grad[B,P n], dsyn[B,nt], flag[B]) in one fused GPU evaluation."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        return self.device_context(param.layer_count(X.shape[1], self.vpvs)).misfit_grad_host(X, which=2)
