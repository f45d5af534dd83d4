"""ctypes binding of librfsurf_b200.so (C ABI declared in include/rfsurfhmc.h)."""
import ctypes as C
import os
import threading
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RFS_LIB") or os.path.join(_HERE, "lib", "librfsurf_b200.so")

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_ubyte)
_i8p = C.POINTER(C.c_byte)
_llp = C.POINTER(C.c_longlong)
_ip = C.POINTER(C.c_int)
_vp = C.c_void_p

WAVETYPES = {"Rc": 0, "Rg": 1, "Lc": 2, "Lg": 3}
PARTYPES = {"rho": 1, "vp": 2, "alpha": 2, "vs": 3, "beta": 3, "h": 4, "thick": 4}


class RfsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[rfs {code}] {msg}")
        self.code = code


_lib = None
_lock = threading.Lock()


def load_library():
    """Load the CUDA library; fails loudly if it was not built (no CPU fallback exists)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). rfsurfhmc_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.rfs_create.restype = C.c_int
        L.rfs_create.argtypes = [C.POINTER(_vp), C.c_int]
        L.rfs_destroy.restype = None
        L.rfs_destroy.argtypes = [_vp]
        L.rfs_last_error.restype = C.c_char_p
        L.rfs_last_error.argtypes = [_vp]
        L.rfs_version.restype = C.c_char_p
        L.rfs_launch_count.restype = C.c_longlong
        L.rfs_launch_count.argtypes = [_vp]
        L.rfs_config_swd.restype = C.c_int
        L.rfs_config_swd.argtypes = [_vp, C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp,
                                     C.c_int, C.c_int, C.c_int]
        L.rfs_config_rf.restype = C.c_int
        L.rfs_config_rf.argtypes = [_vp, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double, C.c_double,
                                    C.c_double, C.c_int, C.c_int]
        L.rfs_config_swd_modes.restype = C.c_int
        L.rfs_config_swd_modes.argtypes = [_vp, C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp,
                                           C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int]
        L.rfs_config_rf_rays.restype = C.c_int
        L.rfs_config_rf_rays.argtypes = [_vp, C.c_int, C.c_int, _dp, C.c_int, C.c_double, C.c_double,
                                         C.c_double, C.c_double, C.c_int, C.c_int]
        L.rfs_config_rf_gauss.restype = C.c_int
        L.rfs_config_rf_gauss.argtypes = [_vp, C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_int, C.c_double,
                                          C.c_double, C.c_double, C.c_int, C.c_int]
        L.rfs_config_obs.restype = C.c_int
        L.rfs_config_obs.argtypes = [_vp, C.c_double, C.c_double, _dp, C.c_int]
        L.rfs_misfit_grad_dev.restype = C.c_int
        L.rfs_misfit_grad_dev.argtypes = [_vp, C.c_longlong, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]
        L.rfs_misfit_grad_host.restype = C.c_int
        L.rfs_misfit_grad_host.argtypes = [_vp, C.c_longlong, _dp, C.c_int, _dp, _dp, _dp, _u8p]
        L.rfs_config_obs_sets.restype = C.c_int
        L.rfs_config_obs_sets.argtypes = [_vp, C.c_int, _dp, _dp, _dp, C.c_int]
        L.rfs_config_obs_rays.restype = C.c_int
        L.rfs_config_obs_rays.argtypes = [_vp, C.c_int, C.c_int, _dp]
        L.rfs_config_obs_periods.restype = C.c_int
        L.rfs_config_obs_periods.argtypes = [_vp, C.c_int, C.c_int, _u8p]
        L.rfs_config_obs_rf_samples.restype = C.c_int
        L.rfs_config_obs_rf_samples.argtypes = [_vp, C.c_int, C.c_int, _u8p]
        L.rfs_config_obs_gauss.restype = C.c_int
        L.rfs_config_obs_gauss.argtypes = [_vp, C.c_int, C.c_int, _dp]
        L.rfs_config_param.restype = C.c_int
        L.rfs_config_param.argtypes = [_vp, C.c_int]
        L.rfs_misfit_grad_sets_dev.restype = C.c_int
        L.rfs_misfit_grad_sets_dev.argtypes = [_vp, C.c_longlong, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]
        L.rfs_misfit_grad_sets_host.restype = C.c_int
        L.rfs_misfit_grad_sets_host.argtypes = [_vp, C.c_longlong, _dp, _ip, C.c_int, _dp, _dp, _dp, _u8p]
        surf_in = [_vp, C.c_longlong, C.c_int, _dp, _dp, _dp, _dp, C.c_int, _dp, C.c_int, C.c_int]
        L.rfs_surf_forward.restype = C.c_int
        L.rfs_surf_forward.argtypes = surf_in + [C.c_int, _dp, _u8p]
        L.rfs_surf_adjoint_kernel.restype = C.c_int
        L.rfs_surf_adjoint_kernel.argtypes = surf_in + [C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _u8p]
        L.rfs_surf_adjoint_kernel_modes.restype = C.c_int
        L.rfs_surf_adjoint_kernel_modes.argtypes = surf_in + [C.c_int, _dp, _dp, _dp, _dp, _dp, _u8p]
        rf_in = [_vp, C.c_longlong, C.c_int] + [_dp] * 6 + [C.c_double, C.c_int, C.c_double, C.c_double,
                                                             C.c_double, C.c_int, C.c_double, C.c_int]
        L.rfs_rf_forward.restype = C.c_int
        L.rfs_rf_forward.argtypes = rf_in + [_dp]
        L.rfs_rf_kernel.restype = C.c_int
        L.rfs_rf_kernel.argtypes = rf_in + [C.c_int, _dp, _dp]
        L.rfs_rf_kernel_all.restype = C.c_int
        L.rfs_rf_kernel_all.argtypes = rf_in + [_dp, _dp]
        L.rfs_hmc_run.restype = C.c_int
        L.rfs_hmc_run.argtypes = [_vp, C.c_int, C.c_int, C.c_longlong, _llp, _dp, C.c_double, C.c_int, C.c_int, C.c_int,
                                  C.c_double, C.c_longlong, C.c_int, C.c_int, C.c_longlong, _dp, _dp, _dp, _dp,
                                  _llp, _llp, _dp, _i8p, C.c_longlong]
        L.rfs_hmc_run_sets.restype = C.c_int
        L.rfs_hmc_run_sets.argtypes = [_vp, C.c_int, C.c_int, C.c_longlong, _llp, _ip, _dp, C.c_int, C.c_double,
                                       C.c_int, C.c_int, C.c_int, C.c_double, C.c_longlong, C.c_int, C.c_int,
                                       C.c_longlong, _dp, _dp, _dp, _dp, _llp, _llp, _dp, _i8p, C.c_longlong]
        L.rfs_hmc_last_evals.restype = C.c_longlong
        L.rfs_hmc_last_evals.argtypes = [_vp]
        L.rfs_hmc_last_steps.restype = C.c_longlong
        L.rfs_hmc_last_steps.argtypes = [_vp]
        L.rfs_set_hmc_options.restype = C.c_int
        L.rfs_set_hmc_options.argtypes = [_vp, C.c_longlong, C.c_double]
        L.rfs_count_evals.restype = C.c_int
        L.rfs_count_evals.argtypes = [_vp, C.c_int]
        L.rfs_read_evals.restype = C.c_longlong
        L.rfs_read_evals.argtypes = [_vp]
        L.rfs_read_eval_stats.restype = C.c_int
        L.rfs_read_eval_stats.argtypes = [_vp, _llp]
        L.rfs_measure_fp64_peak.restype = C.c_int
        L.rfs_measure_fp64_peak.argtypes = [_vp, _dp]
        L.rfs_profile_eval.restype = C.c_int
        L.rfs_profile_eval.argtypes = [_vp, C.c_longlong, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _dp, _llp]
        L.rfs_profile_kernel_name.restype = C.c_char_p
        L.rfs_profile_kernel_name.argtypes = [C.c_int]
        L.rfs_set_roots_team.restype = C.c_int
        L.rfs_set_roots_team.argtypes = [_vp, C.c_int, C.c_int]
        L.rfs_set_roots_sched.restype = C.c_int
        L.rfs_set_roots_sched.argtypes = [_vp, C.c_int]
        L.rfs_last_roots_sched.restype = C.c_int
        L.rfs_last_roots_sched.argtypes = [_vp]
        L.rfs_last_roots_team.restype = C.c_int
        L.rfs_last_roots_team.argtypes = [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.rfs_selftest_math.restype = C.c_int
        L.rfs_selftest_math.argtypes = [_vp, C.c_longlong, _llp]
        _lib = L
        return _lib


def exported_symbols():
    """Every symbol include/rfsurfhmc.h declares (used by the CPU-side ABI test)."""
    return ["rfs_create", "rfs_destroy", "rfs_last_error", "rfs_version", "rfs_launch_count",
            "rfs_config_swd", "rfs_config_rf", "rfs_config_obs", "rfs_misfit_grad_dev",
            "rfs_misfit_grad_host", "rfs_surf_forward", "rfs_surf_adjoint_kernel",
            "rfs_surf_adjoint_kernel_modes", "rfs_rf_forward", "rfs_rf_kernel", "rfs_rf_kernel_all",
            "rfs_hmc_run", "rfs_hmc_last_evals", "rfs_count_evals", "rfs_read_evals",
            "rfs_measure_fp64_peak", "rfs_read_eval_stats", "rfs_selftest_math",
            "rfs_set_roots_team", "rfs_last_roots_team", "rfs_set_roots_sched",
            "rfs_last_roots_sched", "rfs_profile_eval", "rfs_profile_kernel_name",
            "rfs_config_swd_modes", "rfs_config_rf_rays", "rfs_hmc_last_steps", "rfs_set_hmc_options",
            "rfs_config_obs_sets", "rfs_misfit_grad_sets_dev", "rfs_misfit_grad_sets_host", "rfs_hmc_run_sets",
            "rfs_config_obs_rays", "rfs_config_obs_periods", "rfs_config_obs_rf_samples", "rfs_config_rf_gauss",
            "rfs_config_obs_gauss", "rfs_config_param"]


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _sets(sets, rows):
    """Observation-set index per row (int32, host) or None."""
    if sets is None:
        return None
    s = np.ascontiguousarray(np.asarray(sets), dtype=np.int32)
    if s.shape != (rows,):
        raise ValueError(f"sets must have shape ({rows},), got {s.shape}")
    return s


class Context:
    """One opaque rfs_ctx (device workspace + configuration) on one GPU."""

    def __init__(self, device=0):
        self.L = load_library()
        h = _vp()
        rc = self.L.rfs_create(C.byref(h), int(device))
        if rc != 0:
            raise RfsError(rc, "rfs_create failed: no usable CUDA device (rfsurfhmc_b200 has no CPU fallback)")
        self.h = h
        self.device = int(device)
        self.n = None
        self.nt_rf = 0
        self.n_swd_data = 0
        self.nsets = 0
        self.nray = 0
        self.ngauss = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.rfs_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise RfsError(rc, self.L.rfs_last_error(self.h).decode())
        return rc

    def last_error(self):
        return self.L.rfs_last_error(self.h).decode()

    @property
    def launches(self):
        return int(self.L.rfs_launch_count(self.h))

    def count_evals(self, enable=True):
        self._ck(self.L.rfs_count_evals(self.h, int(bool(enable))))

    def read_evals(self):
        return int(self.L.rfs_read_evals(self.h))

    def read_eval_stats(self):
        v = (C.c_longlong * 3)()
        self._ck(self.L.rfs_read_eval_stats(self.h, v))
        return int(v[0]), int(v[1]), int(v[2])

    def set_roots_team(self, T=-1, S=1):
        """Pin the root-search mapping: T<0 automatic, 0 thread-mapped, else T lanes per sequence with
        S speculative scan points (results are bit-identical for every mapping)."""
        self._ck(self.L.rfs_set_roots_team(self.h, int(T), int(S)))

    def set_roots_sched(self, mode=-1):
        """Length-sorted job order of the thread-mapped root search: -1 automatic (large batches), 0 off,
        1 on.  Results are bit-identical either way."""
        self._ck(self.L.rfs_set_roots_sched(self.h, int(mode)))

    def last_roots_sched(self):
        return bool(self.L.rfs_last_roots_sched(self.h))

    def last_roots_team(self):
        t, s = C.c_int(0), C.c_int(0)
        self._ck(self.L.rfs_last_roots_team(self.h, C.byref(t), C.byref(s)))
        return int(t.value), int(s.value)

    def selftest_math(self, n=1 << 22):
        """Mismatch counts (exp, sin/cos large, sin/cos small, rsqrt) of the constant-bank math of the
        root search against the CUDA math library; all zero = bit-identical."""
        v = (C.c_longlong * 6)()
        self._ck(self.L.rfs_selftest_math(self.h, int(n), v))
        return [int(x) for x in v]

    def measure_fp64_peak(self):
        v = C.c_double(0.0)
        self._ck(self.L.rfs_measure_fp64_peak(self.h, C.byref(v)))
        return float(v.value)

    # ---- configuration
    def config_swd(self, nlayer, tRc=None, tRg=None, tLc=None, tLg=None, mode=0, sphere=False, stale=True):
        """mode: int (the reference's SurfWD.mode) or an ascending list of modes (one objective over
        several modes; data vector [mode][Rc,Rg,Lc,Lg])."""
        per = [_f64(t if t is not None else []) for t in (tRc, tRg, tLc, tLg)]
        modes = np.ascontiguousarray(np.atleast_1d(mode), dtype=np.int32)
        self._ck(self.L.rfs_config_swd_modes(
            self.h, int(nlayer), per[0].size, _p(per[0]), per[1].size, _p(per[1]), per[2].size, _p(per[2]),
            per[3].size, _p(per[3]), modes.size, modes.ctypes.data_as(C.POINTER(C.c_int)),
            int(bool(sphere)), int(bool(stale))))
        self.n = int(nlayer)
        self.n_swd_data = sum(p.size for p in per) * modes.size

    def config_rf(self, nlayer, ray_p, nt, dt, gauss, time_shift, water=0.001, rf_type="P", method="freq"):
        """ray_p: float (the reference's ReceiverFunc.ray_p) or a list (one objective over several ray
        parameters; data vector [ray parameter][nt]).  gauss: float (the reference's ReceiverFunc.gauss)
        or a list of Gaussian widths (one objective over all of them; data vector [ray][gauss][nt])."""
        rays = _f64(np.atleast_1d(ray_p))
        if np.ndim(gauss) == 0:
            self._ck(self.L.rfs_config_rf_rays(self.h, int(nlayer), rays.size, _p(rays), int(nt), float(dt),
                                               float(gauss), float(time_shift), float(water),
                                               rf_type_code(rf_type), method_code(method)))
            ng = 1
        else:
            g = _f64(gauss)
            if g.ndim != 1:
                raise ValueError(f"gauss must be a number or a list of widths, got shape {g.shape}")
            self._ck(self.L.rfs_config_rf_gauss(self.h, int(nlayer), rays.size, _p(rays), g.size, _p(g), int(nt),
                                                float(dt), float(time_shift), float(water),
                                                rf_type_code(rf_type), method_code(method)))
            ng = g.size
        self.n = int(nlayer)
        self.nt_rf = int(nt) * rays.size * ng
        self.nray = rays.size
        self.ngauss = ng

    def config_obs(self, dobs, sigma1=1.0, sigma2=1.0):
        """dobs [ndata]: one data vector.  dobs [S, ndata]: S observation sets (stations) sharing the
        forward configuration, with sigma1 / sigma2 scalars or [S] arrays; the evaluations and the HMC
        then take a set index per row / per chain."""
        d = _f64(dobs)
        if d.ndim not in (1, 2) or d.size == 0:
            raise ValueError(f"dobs must be [ndata] or [S, ndata], got shape {d.shape}")
        S = 1 if d.ndim == 1 else d.shape[0]
        s1 = _f64(np.broadcast_to(np.asarray(sigma1, dtype=np.float64), (S,)))
        s2 = _f64(np.broadcast_to(np.asarray(sigma2, dtype=np.float64), (S,)))
        self._ck(self.L.rfs_config_obs_sets(self.h, S, _p(s1), _p(s2), _p(d), d.shape[-1]))
        self.nsets = S

    def config_obs_rays(self, ray_p):
        """Per-station ray parameters: ray_p [S] (one ray parameter per objective) or [S, nray], for the S
        observation sets held now.  Row b then uses ray_p[set[b]] in place of config_rf's shared list.
        config_obs and config_rf drop the table again."""
        r = _f64(ray_p)
        if r.ndim not in (1, 2) or r.shape[0] == 0:
            raise ValueError(f"ray_p must be [S] or [S, nray], got shape {r.shape}")
        nray = 1 if r.ndim == 1 else r.shape[1]
        self._ck(self.L.rfs_config_obs_rays(self.h, r.shape[0], nray, _p(r)))

    def config_obs_periods(self, use):
        """Per-station SWD period lists: use [S, nper] (bool or 0/1) marks the periods of config_swd's
        lists (the common grid, nper = len(tRc) + len(tRg) + len(tLc) + len(tLg), in the data vector's
        order; the same mask for every mode block) that each of the S observation sets held now observes.
        Row b then equals a one-station context configured on set[b]'s subset lists; dsyn is NaN at the
        periods it does not observe.  config_obs and config_swd drop the table again."""
        u = np.asarray(use)
        if u.ndim != 2 or u.shape[0] == 0:
            raise ValueError(f"use must be [S, nper], got shape {u.shape}")
        if u.dtype != np.bool_ and not np.all((u == 0) | (u == 1)):
            raise ValueError("use must hold booleans or 0/1")
        u8 = np.ascontiguousarray(u, dtype=np.uint8)
        self._ck(self.L.rfs_config_obs_periods(self.h, u8.shape[0], u8.shape[1], u8.ctypes.data_as(_u8p)))

    def config_obs_rf_samples(self, use):
        """Per-station receiver-function samples: use [S, nray * ngauss * nt], [S, nray, nt] or
        [S, nray, ngauss, nt] (bool or 0/1) marks the samples of the RF block of the data vector (order
        [ray][gauss][sample]) that each of the S
        observation sets held now fits.  The misfit sums over the observed samples only and dobs is never
        read at the others (NaN there is harmless); dsyn keeps the full traces.  config_obs and config_rf
        drop the table again."""
        u = np.asarray(use)
        if u.ndim not in (2, 3, 4) or u.shape[0] == 0:
            raise ValueError(f"use must be [S, nray * ngauss * nt], [S, nray, nt] or [S, nray, ngauss, nt], "
                             f"got shape {u.shape}")
        if u.dtype != np.bool_ and not np.all((u == 0) | (u == 1)):
            raise ValueError("use must hold booleans or 0/1")
        u8 = np.ascontiguousarray(u.reshape(u.shape[0], -1), dtype=np.uint8)
        self._ck(self.L.rfs_config_obs_rf_samples(self.h, u8.shape[0], u8.shape[1], u8.ctypes.data_as(_u8p)))

    def config_obs_gauss(self, gauss):
        """Per-station Gaussian widths: gauss [S] (one width per objective) or [S, ngauss], for the S
        observation sets held now.  Row b's trace of width g is then deconvolved with gauss[set[b]][g] in
        place of config_rf's shared width g; the data vector keeps its layout.  config_obs and config_rf
        drop the table again."""
        g = _f64(gauss)
        if g.ndim not in (1, 2) or g.shape[0] == 0:
            raise ValueError(f"gauss must be [S] or [S, ngauss], got shape {g.shape}")
        ng = 1 if g.ndim == 1 else g.shape[1]
        self._ck(self.L.rfs_config_obs_gauss(self.h, g.shape[0], ng, _p(g)))

    def config_param(self, vpvs):
        """Model-vector layout of every evaluation and HMC run on this context: vpvs False (default)
        x = [vs, thk] with Brocher vp and rho, True x = [vs, thk, vpvs] with vp = vpvs * vs and Brocher rho
        of that vp.  Accepts a bool or the RFS_PARAM_* code (0, 1)."""
        code = int(vpvs) if not isinstance(vpvs, bool) else (1 if vpvs else 0)
        self._ck(self.L.rfs_config_param(self.h, code))

    def ndata(self, which=0):
        return (self.nt_rf if which != 2 else 0) + (self.n_swd_data if which != 1 else 0)

    # ---- hot path
    def misfit_grad_host(self, x, which=0, sets=None):
        """sets [B]: observation set of each row (required when the context holds several)."""
        x = _f64(x)
        B, n2 = x.shape
        s = _sets(sets, B)
        nd = self.ndata(which)
        U = np.empty(B)
        g = np.empty((B, n2))
        d = np.empty((B, nd))
        f = np.empty(B, dtype=np.uint8)
        self._ck(self.L.rfs_misfit_grad_sets_host(self.h, B, _p(x), s.ctypes.data_as(_ip) if s is not None else None,
                                                  int(which), _p(U), _p(g), _p(d), f.ctypes.data_as(_u8p)))
        return U, g, d, f.astype(bool)

    def misfit_grad_dev(self, B, x_ptr, which, U_ptr, g_ptr, d_ptr, f_ptr, stream_ptr, sets_ptr=0):
        """sets_ptr: device int32 [B] observation set of each row, 0 = none (one set)."""
        self._ck(self.L.rfs_misfit_grad_sets_dev(self.h, int(B), _vp(x_ptr), _vp(sets_ptr or None), int(which),
                                                 _vp(U_ptr), _vp(g_ptr), _vp(d_ptr), _vp(f_ptr), _vp(stream_ptr)))

    PROF_NK = 10

    def profile_eval(self, B, x_ptr, which, U_ptr, g_ptr, d_ptr, f_ptr, stream_ptr):
        """One evaluation with CUDA events around every kernel: {kernel class: (ms, launches)}."""
        ms = (C.c_double * self.PROF_NK)()
        nl = (C.c_longlong * self.PROF_NK)()
        self._ck(self.L.rfs_profile_eval(self.h, int(B), _vp(x_ptr), int(which), _vp(U_ptr), _vp(g_ptr),
                                         _vp(d_ptr), _vp(f_ptr), _vp(stream_ptr), ms, nl))
        return {self.L.rfs_profile_kernel_name(i).decode(): (float(ms[i]), int(nl[i]))
                for i in range(self.PROF_NK)}

    # ---- libsurf / librf drop-ins (batched)
    def surf_forward(self, thk, vp, vs, rho, period, wavetype, mode=0, sphere=False):
        thk, vp, vs, rho = (np.atleast_2d(_f64(a)) for a in (thk, vp, vs, rho))
        t = _f64(period)
        B, n = thk.shape
        c = np.zeros((B, t.size))
        ok = np.zeros(B, dtype=np.uint8)
        self._ck(self.L.rfs_surf_forward(self.h, B, n, _p(thk), _p(vp), _p(vs), _p(rho), t.size, _p(t),
                                         wavetype_code(wavetype), int(mode), int(bool(sphere)), _p(c),
                                         ok.ctypes.data_as(_u8p)))
        return c, ok.astype(bool)

    def surf_adjoint_kernel(self, thk, vp, vs, rho, period, wavetype, mode=0, sphere=False, stale=True,
                            all_modes=False):
        thk, vp, vs, rho = (np.atleast_2d(_f64(a)) for a in (thk, vp, vs, rho))
        t = _f64(period)
        B, n = thk.shape
        nm = (mode + 1) if all_modes else 1
        shp_c = (B, nm, t.size) if all_modes else (B, t.size)
        shp_k = (B, nm, t.size, n) if all_modes else (B, t.size, n)
        c = np.zeros(shp_c)
        da, db, dr, dh = (np.zeros(shp_k) for _ in range(4))
        ok = np.zeros(B, dtype=np.uint8)
        if all_modes:
            self._ck(self.L.rfs_surf_adjoint_kernel_modes(
                self.h, B, n, _p(thk), _p(vp), _p(vs), _p(rho), t.size, _p(t), wavetype_code(wavetype),
                int(mode), int(bool(stale)), _p(c), _p(da), _p(db), _p(dr), _p(dh), ok.ctypes.data_as(_u8p)))
        else:
            self._ck(self.L.rfs_surf_adjoint_kernel(
                self.h, B, n, _p(thk), _p(vp), _p(vs), _p(rho), t.size, _p(t), wavetype_code(wavetype),
                int(mode), int(bool(sphere)), int(bool(stale)), _p(c), _p(da), _p(db), _p(dr), _p(dh),
                ok.ctypes.data_as(_u8p)))
        return c, da, db, dr, dh, ok.astype(bool)

    def _rf_args(self, thk, rho, vp, vs, qa, qb):
        a = [np.atleast_2d(_f64(v)) for v in (thk, rho, vp, vs, qa, qb)]
        return a, a[0].shape

    def rf_forward(self, thk, rho, vp, vs, qa, qb, ray_p, nt, dt, gauss, time_shift, method="time",
                   water=0.001, rf_type="P"):
        a, (B, n) = self._rf_args(thk, rho, vp, vs, qa, qb)
        rf = np.zeros((B, nt))
        self._ck(self.L.rfs_rf_forward(self.h, B, n, *map(_p, a), float(ray_p), int(nt), float(dt),
                                       float(gauss), float(time_shift), method_code(method), float(water),
                                       rf_type_code(rf_type), _p(rf)))
        return rf

    def rf_kernel(self, thk, rho, vp, vs, qa, qb, ray_p, nt, dt, gauss, time_shift, method="time",
                  water=0.001, rf_type="P", par_type="vs"):
        if par_type not in PARTYPES:
            raise ValueError("par_type should be one of [vp,vs,rho,thick]")
        a, (B, n) = self._rf_args(thk, rho, vp, vs, qa, qb)
        rf = np.zeros((B, nt))
        drf = np.zeros((B, n, nt))
        self._ck(self.L.rfs_rf_kernel(self.h, B, n, *map(_p, a), float(ray_p), int(nt), float(dt),
                                      float(gauss), float(time_shift), method_code(method), float(water),
                                      rf_type_code(rf_type), PARTYPES[par_type], _p(rf), _p(drf)))
        return rf, drf

    def rf_kernel_all(self, thk, rho, vp, vs, qa, qb, ray_p, nt, dt, gauss, time_shift, method="time",
                      water=0.001, rf_type="P"):
        a, (B, n) = self._rf_args(thk, rho, vp, vs, qa, qb)
        rf = np.zeros((B, nt))
        drf = np.zeros((B, 4, n, nt))
        self._ck(self.L.rfs_rf_kernel_all(self.h, B, n, *map(_p, a), float(ray_p), int(nt), float(dt),
                                          float(gauss), float(time_shift), method_code(method), float(water),
                                          rf_type_code(rf_type), _p(rf), _p(drf)))
        return rf, drf

    # ---- device-resident HMC
    def set_hmc_options(self, resident=0, max_seconds=0.0):
        """resident > 0: chains share that many device slots (finished chains hand their slot to queued
        ones); max_seconds > 0: wall-clock budget of a run."""
        self._ck(self.L.rfs_set_hmc_options(self.h, int(resident), float(max_seconds)))

    def hmc_run(self, sampler, chain_ids, bounds, dt, Lrange=(5, 20), L0=10, target_ratio=0.65,
                seed=0, nsamples=800, ndraws=200, max_iters=0, want_samples=True, want_syn=False,
                log_accepts=0, which=0, sets=None):
        """bounds [2n, 2] (one box) or [S, 2n, 2] (one box per observation set); sets [C]: observation
        set of each chain (required when the context holds several)."""
        ids = np.ascontiguousarray(np.asarray(chain_ids, dtype=np.int64))
        Cn = ids.size
        s = _sets(sets, Cn)
        b = _f64(bounds)
        if b.ndim not in (2, 3) or b.shape[-1] != 2:
            raise ValueError(f"bounds must be [2n, 2] or [S, 2n, 2], got shape {b.shape}")
        nb = 1 if b.ndim == 2 else b.shape[0]
        n2 = b.shape[-2]
        nd = self.ndata(which)
        out = {
            "misfit": np.zeros((Cn, nsamples)),
            "samples": np.zeros((Cn, nsamples, n2)) if want_samples else None,
            "syn": np.zeros((Cn, nsamples, nd)) if want_syn else None,
            "initmodel": np.zeros((Cn, n2)),
            "n_iter": np.zeros(Cn, dtype=np.int64),
            "n_acc": np.zeros(Cn, dtype=np.int64),
            "dt": np.zeros(Cn),
            "accept_seq": np.zeros((Cn, log_accepts), dtype=np.int8) if log_accepts > 0 else None,
        }
        if Cn == 0:   # a rank without chains (nchains < world size): empty results, nothing to run
            out.update(evals=0, warning="")
            return out
        rc = self.L.rfs_hmc_run_sets(
            self.h, int(sampler), int(which), Cn, ids.ctypes.data_as(_llp),
            s.ctypes.data_as(_ip) if s is not None else None, _p(b), nb, float(dt), int(Lrange[0]),
            int(Lrange[1]), int(L0), float(target_ratio), int(seed), int(nsamples), int(ndraws),
            int(max_iters), _p(out["samples"]), _p(out["misfit"]), _p(out["syn"]), _p(out["initmodel"]),
            out["n_iter"].ctypes.data_as(_llp), out["n_acc"].ctypes.data_as(_llp), _p(out["dt"]),
            out["accept_seq"].ctypes.data_as(_i8p) if log_accepts > 0 else None, int(log_accepts))
        self._ck(rc)
        out["evals"] = int(self.L.rfs_hmc_last_evals(self.h))
        out["global_steps"] = int(self.L.rfs_hmc_last_steps(self.h))
        out["warning"] = self.last_error() if rc > 0 else ""
        return out


def wavetype_code(w):
    if w not in WAVETYPES:
        raise ValueError("wavetype should be one of [Rc,Rg,Lc,Lg]")
    return WAVETYPES[w]


def rf_type_code(t):
    if t in ("P", "p"):
        return 1
    if t in ("S", "s"):
        return 2
    raise ValueError("rf_type should be one of [P,p,S,s]")


def method_code(m):
    return 0 if m == "time" else 1


_default_ctx = {}


def default_context(device=0):
    """Process-wide context used by the per-model drop-in modules (libsurf / librf)."""
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
