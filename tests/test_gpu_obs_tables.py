"""Lifetime of the per-set observation tables (rfs_config_obs_rays, rfs_config_obs_periods and
rfs_config_obs_rf_samples; the rule is stated once in include/rfsurfhmc.h): a table setter that fails
leaves no table of its kind, and a failed rfs_config_swd* or rfs_config_rf* leaves the configuration and
every table as they were."""
import ctypes
import numpy as np
import pytest
from rfsurfhmc_b200._lib import Context
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, perturbed_models

pytestmark = pytest.mark.gpu
RFS_E_ARG, RFS_E_CONFIG = -2, -4
S = 3
CFG = f1_config()
NT = CFG["nt"]
T = np.arange(5., 41.)
_dp = ctypes.POINTER(ctypes.c_double)
_u8p = ctypes.POINTER(ctypes.c_ubyte)
SETTERS = {"rays": "rfs_config_obs_rays", "periods": "rfs_config_obs_periods",
           "rf_samples": "rfs_config_obs_rf_samples"}


def _valid(table):
    """A table that changes every station's misfit.  The period mask observes other Rc than Rg periods at
    station 0, so that the table runs its own plan without the Rc/Rg sequence sharing."""
    if table == "rays":
        return np.array([[0.041], [0.05], [0.058]])
    use = np.ones((S, 2 * T.size if table == "periods" else NT), dtype=np.uint8)
    use[0, :5] = 0
    use[1, -20:] = 0
    use[2, 10:30] = 0
    return use


def _invalid(table):
    """One failing call per error class the header lists for the setter: (S, width, table, code)."""
    good = _valid(table)
    w = good.shape[1]
    cases = [(S - 1, w, good[:S - 1], RFS_E_CONFIG), (S, w, None, RFS_E_ARG)]
    if table == "rays":
        cases.append((S, 2, np.hstack((good, good)), RFS_E_ARG))
        for v in (np.nan, np.inf, 0.0, -0.05):
            bad = good.copy()
            bad[1, 0] = v
            cases.append((S, w, bad, RFS_E_ARG))
        return cases
    cases.append((S, w - 1, good[:, 1:], RFS_E_ARG))
    bad = good.copy()
    bad[1, 3] = 2
    cases.append((S, w, bad, RFS_E_ARG))
    bad = good.copy()
    bad[2] = 0  # a station that observes nothing
    cases.append((S, w, bad, RFS_E_ARG))
    return cases


def _set(c, table, arr, S_=S, width=None):
    """The raw setter call (arr None passes NULL)."""
    a = None if arr is None else np.ascontiguousarray(arr, dtype=np.float64 if table == "rays" else np.uint8)
    ptr = None if a is None else a.ctypes.data_as(_dp if table == "rays" else _u8p)
    return getattr(c.L, SETTERS[table])(c.h, S_, a.shape[1] if width is None else width, ptr)


def _context():
    """The F1 joint objective (Rc and Rg on one grid, one ray parameter) over S stations."""
    c = Context(0)
    c.config_swd(7, T, T.copy())
    c.config_rf(7, CFG["ray_p"], NT, CFG["dt"], CFG["gauss"], CFG["time_shift"], CFG["water"])
    c.config_obs(np.zeros((S, c.ndata())))
    _, _, d, _ = c.misfit_grad_host(perturbed_models(f1_true_model(), S, seed=3), sets=np.arange(S))
    d = np.where(np.isfinite(d), d, 0.0) + 0.01 * np.random.default_rng(3).standard_normal(d.shape)
    c.config_obs(d, [1.0, 0.5, 2.0], [1.0, 1.5, 0.25])
    return c


def _rows(B=48):
    return perturbed_models(f1_true_model(), B, seed=8, rel=0.1), np.arange(B, dtype=np.int32) % S


def _assert_same(got, want, tag):
    for name, a, b in zip(("U", "grad", "dsyn", "flag"), got, want):
        assert np.array_equal(a, b, equal_nan=True), (tag, name)


@pytest.mark.parametrize("table", list(SETTERS))
def test_failed_setter_leaves_no_table(table):
    X, sets = _rows()
    c = _context()
    try:
        plain = c.misfit_grad_host(X, 0, sets=sets)
        for i, (S_, width, arr, code) in enumerate(_invalid(table)):
            assert _set(c, table, _valid(table)) == 0
            assert not np.array_equal(c.misfit_grad_host(X, 0, sets=sets)[0], plain[0])
            assert _set(c, table, arr, S_, width) == code, (table, i)
            _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, (table, i))
    finally:
        c.close()


@pytest.mark.parametrize("call", ["swd_descending_periods", "rf_bad_rf_type"])
def test_failed_configuration_keeps_every_table(call):
    X, sets = _rows()
    c = _context()
    try:
        for table in SETTERS:
            assert _set(c, table, _valid(table)) == 0
        before = c.misfit_grad_host(X, 0, sets=sets)
        if call == "swd_descending_periods":
            t = np.ascontiguousarray(T[::-1])
            tp = t.ctypes.data_as(_dp)
            rc = c.L.rfs_config_swd(c.h, 7, t.size, tp, t.size, tp, 0, None, 0, None, 0, 0, 1)
        else:  # rf_type 3 is neither P nor S; the other arguments differ from the configuration held
            r = np.array([0.05, 0.06])
            rc = c.L.rfs_config_rf_rays(c.h, 7, r.size, r.ctypes.data_as(_dp), 2 * NT, CFG["dt"], CFG["gauss"],
                                        CFG["time_shift"], CFG["water"], 3, 1)
        assert rc == RFS_E_ARG
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), before, call)
    finally:
        c.close()
