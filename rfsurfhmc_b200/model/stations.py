"""StationArray — many stations (observation sets) that share one forward configuration.

A station array is inverted station by station: each station has its own data vector (receiver
function and dispersion curves), its own sigma1 / sigma2 and optionally its own ray parameter(s), its
own subset of the dispersion periods, its own receiver-function samples and its own Gaussian width(s),
while the layer count, the period grid, modes, the width count and RF sampling are shared.  The reference runs one job per station; here one context holds every station's
observations and each evaluated row, or each HMC chain, names its station, so one device run fills the
GPU with all of them (include/rfsurfhmc.h: rfs_config_obs_sets, rfs_config_obs_rays,
rfs_config_obs_periods, rfs_config_obs_rf_samples, rfs_config_obs_gauss).

    stations = StationArray(joint_model, dobs, ray_p=p)   # dobs [S, ndata], p [S] or [S, nray]
    HamitonianMC(stations, bounds, ...).sample_chains(ids, stations=station_of_each_chain)

With swd_use [S, nper] the template's four period lists are a common grid (nper = len(tRc) + len(tRg) +
len(tLc) + len(tLg)) and station s observes the grid periods where swd_use[s] is true: dobs keeps the grid
layout (its values at unobserved periods are ignored), synthetics are NaN there.

With rf_use [S, nray * ngauss * nt] (or [S, nray, ngauss, nt], or [S, nray, nt] with one Gaussian width)
station s fits the receiver-function samples where rf_use[s] is true: a missing ray-parameter bin is a ray
whose traces are all false, a fitting window a run of true samples.  dobs keeps the full layout (its values at unobserved samples are never read, NaN is
fine) and the synthetics keep the full traces.  rf_time_window builds the mask from bounds in seconds.

With gauss [S] or [S, ngauss] station s's receiver functions are computed with its own Gaussian widths
(those its data were processed with) in place of the template's, one per template width: the width count
stays shared, and a station that fits fewer widths drops the others with rf_use.

A stations file (load_stations, `driver --stations`) is an .npz with dobs [S, ndata] and the optional
keys names [S], sigma1 / sigma2 [S], bounds [S, 2n, 2] ([S, 3n, 2] for a template with vpvs=True),
ray_p [S] or [S, nray], swd_use [S, nper], rf_use in one of the shapes above and gauss [S] or [S, ngauss].

The array inherits the template's parameterisation (model/param.py): with vpvs=True every row is
[vs, thk, vpvs] and station_model(s) keeps the flag.
"""
import copy
import numpy as np
from .._lib import Context
from .model_rf_swd_vs_thk import Joint_RF_SWD
from .model_rf import ReceiverFunc
from .model_surf import SurfWD
from . import param


def _fresh_copy(m):
    """Shallow copy of a model object without its device context."""
    c = copy.copy(m)
    c._ctx = None
    c._ctx_key = None
    return c


class StationArray:
    def __init__(self, model, dobs, sigma1=None, sigma2=None, names=None, ray_p=None, swd_use=None,
                 rf_use=None, gauss=None):
        """model: a configured Joint_RF_SWD, ReceiverFunc or SurfWD; only its forward configuration is
        used (its own observations are ignored).  dobs [S, ndata] in the model's data layout.
        sigma1 / sigma2: scalars or [S] (default: the joint model's own, 1.0 for the others; they only
        weight the joint objective).  names [S]: output sub-directories (default station0000, ...).
        ray_p: None (every station uses the template's ray parameter(s)) or each station's own, [S] or
        [S, nray] with the template's ray count; not for a SurfWD template.
        swd_use: None (every station observes every period) or [S, nper] bool / 0-1, the grid periods
        each station observes; for a Joint_RF_SWD or SurfWD template.
        rf_use: None (every station fits every RF sample) or [S, nray * ngauss * nt] / [S, nray, ngauss, nt]
        ([S, nray, nt] with one width) bool / 0-1, the receiver-function samples each station fits (see
        rf_time_window); for a Joint_RF_SWD or ReceiverFunc template.
        gauss: None (every station uses the template's Gaussian width(s)) or each station's own, [S] or
        [S, ngauss] with the template's width count; not for a SurfWD template."""
        if not (hasattr(model, "_config_forward") and hasattr(model, "which")):
            raise TypeError("StationArray needs a Joint_RF_SWD, ReceiverFunc or SurfWD template")
        self.template = model
        self.which = model.which
        self.dobs = np.array(dobs, dtype=np.float64, ndmin=2)
        if self.dobs.ndim != 2:
            raise ValueError(f"dobs must be [S, ndata], got shape {self.dobs.shape}")
        S, nd = self.dobs.shape
        want = model.ndata if isinstance(model, Joint_RF_SWD) else model.nt
        if nd != want:
            raise ValueError(f"dobs has {nd} values per station, the model's data vector has {want}")
        self.nstations = S
        self.ndata = nd
        s1 = getattr(model, "sigma1", 1.0) if sigma1 is None else sigma1
        s2 = getattr(model, "sigma2", 1.0) if sigma2 is None else sigma2
        self.sigma1 = np.broadcast_to(np.asarray(s1, dtype=np.float64), (S,)).copy()
        self.sigma2 = np.broadcast_to(np.asarray(s2, dtype=np.float64), (S,)).copy()
        self.names = [f"station{s:04d}" for s in range(S)] if names is None else [str(v) for v in names]
        if len(self.names) != S:
            raise ValueError(f"names has {len(self.names)} entries for {S} stations")
        self.ray_p = None
        if ray_p is not None:
            rf = model.rfmodel if isinstance(model, Joint_RF_SWD) else model
            if not isinstance(rf, ReceiverFunc):
                raise TypeError("ray_p needs a receiver-function template (Joint_RF_SWD or ReceiverFunc)")
            self.ray_p = station_rays(ray_p, S, rf.nray)
        self.swd_use = None
        if swd_use is not None:
            swd = model.swdmodel if isinstance(model, Joint_RF_SWD) else model
            if not isinstance(swd, SurfWD):
                raise TypeError("swd_use needs a dispersion template (Joint_RF_SWD or SurfWD)")
            self.swd_use = station_periods(swd_use, S, swd)
        self.rf_use = None
        if rf_use is not None:
            rf = model.rfmodel if isinstance(model, Joint_RF_SWD) else model
            if not isinstance(rf, ReceiverFunc):
                raise TypeError("rf_use needs a receiver-function template (Joint_RF_SWD or ReceiverFunc)")
            self.rf_use = station_rf_samples(rf_use, S, rf)
        self.gauss = None
        if gauss is not None:
            rf = model.rfmodel if isinstance(model, Joint_RF_SWD) else model
            if not isinstance(rf, ReceiverFunc):
                raise TypeError("gauss needs a receiver-function template (Joint_RF_SWD or ReceiverFunc)")
            self.gauss = station_gauss(gauss, S, rf.ngauss)
        self._ctx = None
        self._ctx_key = None

    @property
    def _device(self):
        return self.template._device

    @property
    def vpvs(self):
        return self.template.vpvs

    @property
    def npar(self):
        return param.npar(self.vpvs)

    def device_context(self, n):
        """Configured rfs context (the template's forward configuration + every station's observations)
        for n layers; re-configured whenever a template field, a sigma or an observation has changed."""
        if self._ctx is None or self._ctx.device != self._device:
            self._ctx = Context(self._device)
            self._ctx_key = None
        key = (type(self.template), self.template._config_fields(n), self.sigma1.tobytes(),
               self.sigma2.tobytes(), self.dobs.tobytes(), None if self.ray_p is None else self.ray_p.tobytes(),
               None if self.swd_use is None else self.swd_use.tobytes(),
               None if self.rf_use is None else self.rf_use.tobytes(),
               None if self.gauss is None else self.gauss.tobytes())
        if self._ctx_key != key:
            self.template._config_forward(self._ctx, n)
            self._ctx.config_obs(self.dobs, self.sigma1, self.sigma2)
            if self.ray_p is not None:
                self._ctx.config_obs_rays(self.ray_p)
            if self.swd_use is not None:
                self._ctx.config_obs_periods(self.swd_use)
            if self.rf_use is not None:
                self._ctx.config_obs_rf_samples(self.rf_use)
            if self.gauss is not None:
                self._ctx.config_obs_gauss(self.gauss)
            self._ctx_key = key
        return self._ctx

    def misfit_and_grad_batch(self, X, stations):
        """X [B, P n], stations [B] -> (U[B], grad[B,P n], dsyn[B,ndata], flag[B]): row b against station
        stations[b], all rows in one fused GPU evaluation."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        return self.device_context(param.layer_count(X.shape[1], self.vpvs)).misfit_grad_host(
            X, which=self.which, sets=stations)

    def station_model(self, s):
        """Single-station copy of the template holding station s's observations (and sigmas, ray
        parameter(s): a scalar for one ray, a list otherwise, and Gaussian width(s): a scalar when the
        template's gauss is one, a list otherwise).  With swd_use its SurfWD holds the
        station's subset period lists and its dispersion data only the observed values.  With rf_use its
        ReceiverFunc holds only the station's observed rays and widths (ray parameters, widths and
        traces); a station that fits part of a trace, or whose observed traces are not every observed
        width of every observed ray, has no single-station model (ValueError)."""
        s = int(s)
        if not 0 <= s < self.nstations:
            raise IndexError(f"station {s} outside [0, {self.nstations})")
        d = self.dobs[s].copy()
        t = self.template
        if isinstance(t, Joint_RF_SWD):
            rf, keep = self._station_rf(t.rfmodel, s)
            m = Joint_RF_SWD(float(self.sigma1[s]), float(self.sigma2[s]), rf, self._station_swd(t.swdmodel, s))
            m._device = t._device
            nt = t.rfmodel.nt
            m.set_obsdata(d[:nt][keep], self._compact(d[nt:], s))
            return m
        if isinstance(t, ReceiverFunc):
            m, keep = self._station_rf(t, s)
            d = d[keep]
        else:
            m = self._station_swd(t, s)
            d = self._compact(d, s)
        m.set_obsdata(d)
        return m

    def station_view(self, s):
        """Station s in the array's own data layout: .dobs [ndata] and .misfit_and_grad(x) through the
        grouped context (dsyn NaN at the periods the station does not observe)."""
        return _StationView(self, int(s))

    def _compact(self, dswd, s):
        if self.swd_use is None:
            return dswd
        nmode = dswd.size // self.swd_use.shape[1]
        return dswd[np.tile(self.swd_use[s], nmode)]

    def _station_swd(self, swd, s):
        c = _fresh_copy(swd)
        if self.swd_use is None:
            return c
        u = self.swd_use[s]
        o = 0
        nt = 0
        for w in ("Rc", "Rg", "Lc", "Lg"):
            k = getattr(swd, "nt" + w)
            if k:
                t = np.asarray(getattr(swd, "t" + w))[u[o:o + k]]
                setattr(c, "t" + w, t if t.size else None)
                setattr(c, "nt" + w, int(t.size))
                nt += t.size
                o += k
        c.nt = nt * swd.nmode
        return c

    def _station_rf(self, rf, s):
        """Station s's ReceiverFunc and the data positions of its observed traces."""
        c = _fresh_copy(rf)
        r = self.ray_p[s] if self.ray_p is not None else np.atleast_1d(np.asarray(rf.ray_p, dtype=np.float64))
        keep = np.ones(rf.nt, dtype=bool)
        widths = np.ones(rf.ngauss, dtype=bool)
        if self.rf_use is not None:
            u = self.rf_use[s].reshape(rf.nray, rf.ngauss, rf.nt_trace)
            obs = u.all(axis=2)
            if not np.array_equal(obs, u.any(axis=2)):
                raise ValueError(f"station {s} ({self.names[s]}) fits part of a receiver-function trace: no "
                                 "single-station ReceiverFunc fits a window, use station_view")
            # a ReceiverFunc evaluates every width of every ray: the observed traces must be such a product
            rays, widths = obs.any(axis=1), obs.any(axis=0)
            if not np.array_equal(obs, np.outer(rays, widths)):
                raise ValueError(f"station {s} ({self.names[s]}) observes different Gaussian widths on different "
                                 "rays: no single-station ReceiverFunc fits that, use station_view")
            r = r[rays]
            keep = u.reshape(-1)
            c.nray = int(r.size)
            c.ngauss = int(widths.sum())
            c.nt = c.nt_trace * c.nray * c.ngauss
        if self.ray_p is not None or self.rf_use is not None:
            c.ray_p = float(r[0]) if r.size == 1 else r.tolist()
        # the station's own widths, or the template's observed ones; a template scalar stays a scalar
        if self.gauss is not None or (self.rf_use is not None and np.ndim(rf.gauss) > 0):
            g = (self.gauss[s] if self.gauss is not None else np.asarray(rf.gauss, dtype=np.float64))[widths]
            c.gauss = float(g[0]) if np.ndim(rf.gauss) == 0 else g.tolist()
        return c, keep


class _StationView:
    def __init__(self, array, s):
        self._array, self._s = array, s
        self.dobs = array.dobs[s]

    def misfit_and_grad(self, x):
        U, g, d, f = self._array.misfit_and_grad_batch(np.asarray(x, dtype=np.float64)[None, :], [self._s])
        return U[0], g[0], d[0], bool(f[0])


def station_periods(use, S, swd, where=""):
    """swd_use [S, nper] (bool or 0/1) of a SurfWD template's period grid -> bool [S, nper]; the
    ValueError names the key 'swd_use' (after `where`)."""
    nper = swd.ntRc + swd.ntRg + swd.ntLc + swd.ntLg
    u = np.asarray(use)
    if u.shape != (S, nper):
        raise ValueError(f"{where}'swd_use' must have shape [{S}, {nper}], got {u.shape}")
    if u.dtype != np.bool_ and not np.all((u == 0) | (u == 1)):
        raise ValueError(f"{where}'swd_use' must hold booleans or 0/1")
    u = np.ascontiguousarray(u, dtype=bool)
    empty = np.flatnonzero(~u.any(axis=1))
    if empty.size:
        raise ValueError(f"{where}'swd_use': station {int(empty[0])} observes no period")
    # SurfWD evaluates Love waves on tRc (model_surf.py _grad_periods): a station whose Lc / Lg periods
    # differ from its Rc periods has no single-station SurfWD
    rc = u[:, :swd.ntRc]
    o = swd.ntRc + swd.ntRg
    for w, k in (("Lc", swd.ntLc), ("Lg", swd.ntLg)):
        if k and not np.array_equal(u[:, o:o + k], rc):
            bad = int(np.flatnonzero(np.any(u[:, o:o + k] != rc, axis=1))[0])
            raise ValueError(f"{where}'swd_use': station {bad} observes other {w} than Rc periods; SurfWD "
                             f"evaluates Love waves on tRc, so the {w} mask must equal the Rc mask")
        o += k
    return u


def station_rf_samples(use, S, rf, where=""):
    """rf_use [S, nray * ngauss * nt], [S, nray, ngauss, nt] or, with one Gaussian width, [S, nray, nt]
    (bool or 0/1) of a ReceiverFunc template's data vector -> bool [S, nray * ngauss * nt]; the ValueError
    names the key 'rf_use' (after `where`)."""
    u = np.asarray(use)
    shapes = [(S, rf.nt), (S, rf.nray, rf.ngauss, rf.nt_trace)]
    if rf.ngauss == 1:
        shapes.append((S, rf.nray, rf.nt_trace))
    if u.shape not in shapes:
        raise ValueError(f"{where}'rf_use' must have shape " + " or ".join(
            "[" + ", ".join(map(str, sh)) + "]" for sh in shapes) + f", got {u.shape}")
    if u.dtype != np.bool_ and not np.all((u == 0) | (u == 1)):
        raise ValueError(f"{where}'rf_use' must hold booleans or 0/1")
    u = np.ascontiguousarray(u.reshape(S, rf.nt), dtype=bool)
    empty = np.flatnonzero(~u.any(axis=1))
    if empty.size:
        # a station without RF data would get a zero joint weight and lose its dispersion data silently
        raise ValueError(f"{where}'rf_use': station {int(empty[0])} observes no receiver-function sample")
    return u


def rf_time_window(rf, lo, hi):
    """RF sample mask (rf_use) of the time windows lo <= t <= hi on a ReceiverFunc's trace axis
    t = arange(nt) * dt - time_shift (rf.t), in seconds.  lo, hi: [S] (every ray) or [S, nray]; a NaN
    bound marks a ray the station does not observe.  A ray's bounds apply to every Gaussian width of
    that ray.  A bound equal to a sample time, up to rounding (1e-9 of dt), includes that sample.
    Returns bool [S, nray * ngauss * nt]."""
    lo = np.asarray(lo, dtype=np.float64)
    hi = np.asarray(hi, dtype=np.float64)
    if lo.shape != hi.shape or lo.ndim not in (1, 2) or (lo.ndim == 2 and lo.shape[1] != rf.nray):
        raise ValueError(f"lo and hi must both be [S] or [S, {rf.nray}], got {lo.shape} and {hi.shape}")
    S = lo.shape[0]
    lo = np.broadcast_to(lo.reshape(S, -1), (S, rf.nray))
    hi = np.broadcast_to(hi.reshape(S, -1), (S, rf.nray))
    eps = 1e-9 * rf.dt
    t = np.asarray(rf.t, dtype=np.float64)
    # comparisons with NaN are false: a NaN bound leaves its ray without samples
    u = (t >= lo[..., None] - eps) & (t <= hi[..., None] + eps)
    u = np.broadcast_to(u[:, :, None, :], (S, rf.nray, rf.ngauss, rf.nt_trace))
    return np.ascontiguousarray(u.reshape(S, rf.nt))


def station_rays(ray_p, S, nray, where=""):
    """ray_p [S] (nray = 1) or [S, nray] -> float64 [S, nray], finite and > 0; the ValueError names the
    key 'ray_p' (after `where`)."""
    r = np.asarray(ray_p, dtype=np.float64)
    if not (r.shape == (S, nray) or (nray == 1 and r.shape == (S,))):
        want = f"[{S}] or [{S}, 1]" if nray == 1 else f"[{S}, {nray}]"
        raise ValueError(f"{where}'ray_p' must have shape {want}, got {r.shape}")
    if not np.all(np.isfinite(r) & (r > 0)):
        raise ValueError(f"{where}'ray_p' must be finite and positive")
    return np.ascontiguousarray(r.reshape(S, nray))


def station_gauss(gauss, S, ngauss, where=""):
    """gauss [S] (ngauss = 1) or [S, ngauss] -> float64 [S, ngauss], finite and > 0; the ValueError names
    the key 'gauss' (after `where`)."""
    g = np.asarray(gauss, dtype=np.float64)
    if not (g.shape == (S, ngauss) or (ngauss == 1 and g.shape == (S,))):
        want = f"[{S}] or [{S}, 1]" if ngauss == 1 else f"[{S}, {ngauss}]"
        raise ValueError(f"{where}'gauss' must have shape {want}, got {g.shape}")
    if not np.all(np.isfinite(g) & (g > 0)):
        raise ValueError(f"{where}'gauss' must be finite and positive")
    return np.ascontiguousarray(g.reshape(S, ngauss))


def load_stations(src, ndata, nparam, default_bounds, nray=1, swd=None, rf=None, ngauss=1):
    """Validated content of a stations file (.npz path or a mapping with the same keys):
    dobs [S, ndata] (required), names [S], sigma1 / sigma2 [S] (default 1.0), bounds [S, nparam, 2]
    (default: default_bounds [nparam, 2] for every station), ray_p [S] or [S, nray] (default None: the
    ray parameter(s) of the forward configuration), swd_use [S, nper] (default None: every period;
    swd = the SurfWD whose period grid it marks) and rf_use [S, nray * ngauss * nt] or
    [S, nray, ngauss, nt] ([S, nray, nt] with one width; default None: every RF sample; rf = the
    ReceiverFunc whose data it marks) and gauss [S] or [S, ngauss] (default None: the Gaussian width(s)
    of the forward configuration).  Raises ValueError naming the bad key."""
    if isinstance(src, (str, bytes)) or hasattr(src, "__fspath__"):
        with np.load(src, allow_pickle=False) as f:
            src = {k: f[k] for k in f.files}
    if "dobs" not in src:
        raise ValueError("stations file: key 'dobs' [S, ndata] is required")
    dobs = np.asarray(src["dobs"], dtype=np.float64)
    if dobs.ndim != 2 or dobs.shape[0] < 1 or dobs.shape[1] != ndata:
        raise ValueError(f"stations file: 'dobs' must have shape [S, {ndata}], got {dobs.shape}")
    S = dobs.shape[0]
    out = {"dobs": dobs}
    names = np.asarray(src["names"]) if "names" in src else np.array([f"station{s:04d}" for s in range(S)])
    if names.shape != (S,):
        raise ValueError(f"stations file: 'names' must have shape [{S}], got {names.shape}")
    out["names"] = [str(v) for v in names]
    if len(set(out["names"])) != S or any(not v or "/" in v or v in (".", "..") for v in out["names"]):
        raise ValueError("stations file: 'names' must be distinct, non-empty and free of '/'")
    for key in ("sigma1", "sigma2"):
        v = np.asarray(src[key], dtype=np.float64) if key in src else np.ones(S)
        if v.shape != (S,):
            raise ValueError(f"stations file: '{key}' must have shape [{S}], got {v.shape}")
        if not np.all(np.isfinite(v) & (v > 0)):
            raise ValueError(f"stations file: '{key}' must be finite and positive")
        out[key] = v
    if "bounds" in src:
        b = np.asarray(src["bounds"], dtype=np.float64)
        if b.shape != (S, nparam, 2):
            raise ValueError(f"stations file: 'bounds' must have shape [{S}, {nparam}, 2], got {b.shape}")
        if not np.all(b[..., 0] <= b[..., 1]):
            raise ValueError("stations file: 'bounds' needs low <= high in every row")
    else:
        b = np.broadcast_to(np.asarray(default_bounds, dtype=np.float64), (S, nparam, 2)).copy()
    out["bounds"] = b
    out["ray_p"] = station_rays(src["ray_p"], S, nray, "stations file: ") if "ray_p" in src else None
    out["swd_use"] = None
    if "swd_use" in src:
        if swd is None:
            raise ValueError("stations file: 'swd_use' needs a dispersion configuration")
        out["swd_use"] = station_periods(src["swd_use"], S, swd, "stations file: ")
    out["rf_use"] = None
    if "rf_use" in src:
        if rf is None:
            raise ValueError("stations file: 'rf_use' needs a receiver-function configuration")
        out["rf_use"] = station_rf_samples(src["rf_use"], S, rf, "stations file: ")
    out["gauss"] = station_gauss(src["gauss"], S, ngauss, "stations file: ") if "gauss" in src else None
    return out
