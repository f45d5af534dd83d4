"""Per-station Gaussian widths (rfs_config_obs_gauss): every row of a grouped evaluation, and every chain
of a grouped HMC run, must give exactly what a context holding only that row's station, configured with
that station's widths through config_rf, gives."""
import os
import ctypes
import numpy as np
import pytest
import torch
import yaml
from rfsurfhmc_b200._lib import Context, RfsError
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RFS_E_ARG, RFS_E_CONFIG = -2, -4
S = 5
SIGMA1 = np.array([1.0, 0.5, 2.0, 1.0, 0.8])
SIGMA2 = np.array([1.0, 1.5, 1.0, 0.25, 1.0])
G1 = np.array([1.0, 2.5, 2.0, 3.0, 1.0])  # one width per station (template: F1's 1.5)
G2 = np.array([[1.0, 2.5], [1.5, 3.0], [0.5, 2.0], [2.0, 5.0], [1.2, 2.4]])  # template [1.0, 2.5]
RAYS2 = np.array([[0.04, 0.06], [0.045, 0.065], [0.05, 0.07], [0.055, 0.062], [0.042, 0.071]])
T = np.arange(5., 41.)
_dp = ctypes.POINTER(ctypes.c_double)

# (name, which, RF method, RF type, template ray parameter(s), template width(s), per-station table)
CASES = [
    ("joint_freq_one", 0, "freq", "P", 0.045, 1.5, G1),
    ("joint_freq_two", 0, "freq", "P", 0.045, [1.0, 2.5], G2),
    ("rf_freq_two_rays", 1, "freq", "P", [0.04, 0.06], [1.0, 2.5], G2),
    ("joint_time_two", 0, "time", "P", 0.045, [1.0, 2.5], G2),
    ("rf_time_two", 1, "time", "P", 0.045, [1.0, 2.5], G2),
    ("joint_S", 0, "freq", "S", 0.1, 1.5, G1),
    ("rf_S_two", 1, "freq", "S", 0.1, [1.0, 2.5], G2),
]


def _configure(c, which, method="freq", rf_type="P", rays=0.045, gauss=1.5):
    cfg = f1_config()
    if which != 1:
        c.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"])
    if which != 2:
        c.config_rf(7, rays, cfg["nt"], cfg["dt"], gauss, cfg["time_shift"], cfg["water"], rf_type, method)


def _station_widths(table, s, template):
    """Station s's widths in the template's form: a scalar for a scalar template, a list otherwise."""
    g = np.atleast_1d(table[s])
    return float(g[0]) if np.ndim(template) == 0 else g.tolist()


def _stations(c, which, table, nsta=S, seed=3):
    """Observations of nsta stations, each forward-modelled with its own widths: seeded perturbations of
    the F1 true model plus seeded noise (c is configured for the RF objective)."""
    c.config_obs(np.zeros((nsta, c.ndata(which))))
    c.config_obs_gauss(table[:nsta])
    Xs = perturbed_models(f1_true_model(), nsta, seed=seed, rel=0.05)
    _, _, d, _ = c.misfit_grad_host(Xs, which, sets=np.arange(nsta))
    d = np.where(np.isfinite(d), d, 0.0)
    return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)


def _rows(B=333, seed=8, nsta=S):
    """Models near the truth, strongly inverted ones and ones with a slow half-space (about half of
    those fail the root search), each row on a random station; every station appears."""
    x0 = f1_true_model()
    X = perturbed_models(x0, B, seed=seed, rel=0.1)
    rng = np.random.default_rng(seed)
    kind = rng.random(B)
    wild = kind < 0.2
    X[wild] = rng.uniform(0.5, 1.5, (int(wild.sum()), x0.size)) * x0 + 0.01
    slow = kind > 0.85
    X[slow, x0.size // 2 - 1] = rng.uniform(1.0, 2.5, int(slow.sum()))
    sets = rng.integers(0, nsta, B).astype(np.int32)
    sets[:nsta] = np.arange(nsta)
    return X, sets


def _per_station(which, method, rf_type, rays, gauss, table, dobs, X, sets, rays_table=None, use=None):
    """Reference: one context per station, configured with that station's widths through config_rf (and
    that station's row of the ray table and of the RF-sample mask, when given), on that station's rows."""
    out = [np.zeros(len(X)), np.zeros(X.shape), None, np.zeros(len(X), dtype=bool)]
    for s in range(len(dobs)):
        c = Context(0)
        try:
            _configure(c, which, method, rf_type, rays, _station_widths(table, s, gauss))
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
            if rays_table is not None:
                c.config_obs_rays(rays_table[s:s + 1])
            if use is not None:
                c.config_obs_rf_samples(use[s:s + 1])
            if out[2] is None:
                out[2] = np.zeros((len(X), c.ndata(which)))
            r = sets == s
            for o, v in zip(out, c.misfit_grad_host(X[r], which)):
                o[r] = v
        finally:
            c.close()
    return out


def _assert_same(got, want, tag, rows=slice(None)):
    for name, a, b in zip(("U", "grad", "dsyn", "flag"), got, want):
        assert np.array_equal(a[rows], b[rows], equal_nan=True), (tag, name)


@pytest.mark.parametrize("name,which,method,rf_type,rays,gauss,table", CASES, ids=[c[0] for c in CASES])
def test_grouped_widths_equal_per_station_contexts(name, which, method, rf_type, rays, gauss, table):
    c = Context(0)
    try:
        _configure(c, which, method, rf_type, rays, gauss)
        dobs = _stations(c, which, table)
        X, sets = _rows()
        c.config_obs(dobs, SIGMA1, SIGMA2)
        shared = c.misfit_grad_host(X, which, sets=sets)
        c.config_obs_gauss(table)
        got = c.misfit_grad_host(X, which, sets=sets)
    finally:
        c.close()
    want = _per_station(which, method, rf_type, rays, gauss, table, dobs, X, sets)
    _assert_same(got, want, name)
    ok = got[3] & shared[3]
    assert not np.array_equal(got[0][ok], shared[0][ok])  # the table is really used
    if which == 0:
        fail = ~got[3]
        assert fail.any() and fail.sum() < len(X) // 2
        # the failure convention returns the row's own station's dobs
        assert np.array_equal(got[2][fail], dobs[sets[fail]])


def _drop_one_width(nt):
    """RF-sample mask [S, 2 rays, 2 widths, nt]: station 1 fits only its second width, station 3 only its
    first, station 4 a window of every trace."""
    use = np.ones((S, 2, 2, nt), dtype=bool)
    use[1, :, 0] = False
    use[3, :, 1] = False
    use[4, :, :, :30] = False
    return use.reshape(S, -1)


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "freq"), (0, "time")])
def test_widths_with_a_ray_table_and_an_rf_sample_mask(which, method):
    rays, gauss = [0.04, 0.06], [1.0, 2.5]
    use = _drop_one_width(f1_config()["nt"])
    c = Context(0)
    try:
        _configure(c, which, method, "P", rays, gauss)
        dobs = _stations(c, which, G2)
        X, sets = _rows(B=200, seed=14)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_rays(RAYS2)
        c.config_obs_rf_samples(use)
        without = c.misfit_grad_host(X, which, sets=sets)
        c.config_obs_gauss(G2)
        got = c.misfit_grad_host(X, which, sets=sets)
    finally:
        c.close()
    ok = got[3] & without[3]
    assert not np.array_equal(got[0][ok], without[0][ok])
    want = _per_station(which, method, "P", rays, gauss, G2, dobs, X, sets, rays_table=RAYS2, use=use)
    _assert_same(got, want, (which, method))


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "time")])
def test_chunked_batch_uses_each_chunks_own_widths(which, method):
    """A 1 MiB workspace budget forces many small chunks: each chunk's RF kernels must read the widths of
    its own rows."""
    gauss = [1.0, 2.5]
    X, sets = _rows()
    plain = Context(0)
    try:
        _configure(plain, which, method, gauss=gauss)
        dobs = _stations(plain, which, G2)
        plain.config_obs(dobs, SIGMA1, SIGMA2)
        plain.config_obs_gauss(G2)
        n0 = plain.launches
        want = plain.misfit_grad_host(X, which, sets=sets)
        plain_launches = plain.launches - n0
    finally:
        plain.close()
    old = os.environ.get("RFS_WS_BUDGET_MB")
    os.environ["RFS_WS_BUDGET_MB"] = "1"
    try:
        c = Context(0)
    finally:
        if old is None:
            del os.environ["RFS_WS_BUDGET_MB"]
        else:
            os.environ["RFS_WS_BUDGET_MB"] = old
    try:
        _configure(c, which, method, gauss=gauss)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_gauss(G2)
        n0 = c.launches
        got = c.misfit_grad_host(X, which, sets=sets)
        assert c.launches - n0 >= 4 * plain_launches  # really chunked
    finally:
        c.close()
    _assert_same(got, want, "chunked")
    _assert_same(got, _per_station(which, method, "P", 0.045, gauss, G2, dobs, X, sets), "chunked vs per station")


@pytest.mark.parametrize("which,method,gauss", [(0, "freq", 1.5), (0, "freq", [1.0, 2.5]), (1, "time", [1.0, 2.5]),
                                                (1, "freq", [1.0, 2.5, 5.0])])
def test_table_of_the_shared_widths_gives_the_same_bits(which, method, gauss):
    c = Context(0)
    try:
        _configure(c, which, method, "P", 0.045, gauss)
        g = np.atleast_1d(gauss)
        c.config_obs(np.zeros((S, c.ndata(which))))
        dobs = _stations(c, which, np.tile(g, (S, 1)))
        X, sets = _rows(B=160, seed=11)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        want = c.misfit_grad_host(X, which, sets=sets)
        c.config_obs_gauss(np.tile(g, (S, 1)))
        got = c.misfit_grad_host(X, which, sets=sets)
    finally:
        c.close()
    _assert_same(got, want, "shared table")


def _dev_eval(c, X, s, which):
    dev = torch.device("cuda", 0)
    xd = torch.from_numpy(X).to(dev)
    sd = torch.from_numpy(s).to(dev)
    U = torch.full((len(X),), 7.0, dtype=torch.float64, device=dev)
    G = torch.full((len(X), X.shape[1]), 7.0, dtype=torch.float64, device=dev)
    D = torch.zeros((len(X), c.ndata(which)), dtype=torch.float64, device=dev)
    F = torch.full((len(X),), 9, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev)
    c.misfit_grad_dev(len(X), xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                      st.cuda_stream, sets_ptr=sd.data_ptr())
    st.synchronize()
    return [U.cpu().numpy(), G.cpu().numpy(), D.cpu().numpy(), F.cpu().numpy()]


@pytest.mark.parametrize("which,method,gauss", [(0, "freq", 1.5), (1, "freq", [1.0, 2.5]), (1, "time", [1.0, 2.5]),
                                                (0, "time", 1.5)])
def test_out_of_range_set_fails_only_its_row(which, method, gauss):
    table = G1 if np.ndim(gauss) == 0 else G2
    c = Context(0)
    try:
        _configure(c, which, method, gauss=gauss)
        dobs = _stations(c, which, table)
        X, sets = _rows(B=96, seed=4)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_gauss(table)
        for bad in (-1, S):
            s = sets.copy()
            s[7] = bad
            with pytest.raises(RfsError) as e:
                c.misfit_grad_host(X, which, sets=s)
            assert e.value.code == RFS_E_ARG
        want = c.misfit_grad_host(X, which, sets=sets)
        s = sets.copy()
        bad = np.array([3, 40, 95])
        s[bad] = [-1, S, 1 << 30]
        got = _dev_eval(c, X, s, which)
        assert (got[0][bad] == 0).all() and (got[1][bad] == 0).all() and np.isnan(got[2][bad]).all()
        assert not got[3][bad].any() and set(got[3].tolist()) <= {0, 1}
        got[3] = got[3].astype(bool)
        _assert_same(got, want, "out of range", np.setdiff1d(np.arange(len(X)), bad))
    finally:
        c.close()


def _raw(c, S_, ngauss, table):
    """The raw setter call (table None passes NULL)."""
    if table is None:
        return c.L.rfs_config_obs_gauss(c.h, S_, ngauss, None)
    t = np.ascontiguousarray(table, dtype=np.float64)
    return c.L.rfs_config_obs_gauss(c.h, S_, ngauss, t.ctypes.data_as(_dp))


def _invalid():
    """One failing call per error class of rfs_config_obs_gauss on a two-width objective:
    (S, ngauss, table, code)."""
    cases = [(S - 1, 2, G2[:S - 1], RFS_E_CONFIG), (S + 1, 2, np.vstack((G2, G2[:1])), RFS_E_CONFIG),
             (S, 2, None, RFS_E_ARG), (S, 1, G2[:, :1], RFS_E_ARG), (S, 3, np.hstack((G2, G2[:, :1])), RFS_E_ARG)]
    for v in (0.0, -1.0, np.nan, np.inf, -np.inf):
        t = G2.copy()
        t[2, 1] = v
        cases.append((S, 2, t, RFS_E_ARG))
    return cases


def test_config_obs_gauss_errors_and_a_failed_call_leaves_no_table():
    c = Context(0)
    try:
        _configure(c, 2)  # SWD only: no RF configuration
        c.config_obs(np.zeros((S, c.ndata(2))))
        assert _raw(c, S, 1, G1[:, None]) == RFS_E_CONFIG
        with pytest.raises(RfsError) as e:
            c.config_obs_gauss(G1)
        assert e.value.code == RFS_E_CONFIG
    finally:
        c.close()
    gauss = [1.0, 2.5]
    X, sets = _rows(B=64, seed=9)
    c = Context(0)
    try:
        _configure(c, 0, gauss=gauss)
        assert _raw(c, S, 2, G2) == RFS_E_CONFIG  # no observation sets yet
        dobs = _stations(c, 0, G2)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        plain = c.misfit_grad_host(X, 0, sets=sets)
        assert _raw(c, S, 2, G2) == 0
        table = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(table[0], plain[0])
        for i, (S_, ng, t, code) in enumerate(_invalid()):
            assert _raw(c, S, 2, G2) == 0
            _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, ("valid", i))
            assert _raw(c, S_, ng, t) == code, i
            _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, ("failed", i))
        with pytest.raises(RfsError) as e:  # the Python wrapper reports the same
            c.config_obs_gauss(G1)
        assert e.value.code == RFS_E_ARG
    finally:
        c.close()


def test_config_calls_drop_or_keep_the_table():
    """Call by call: rfs_config_obs_sets, rfs_config_obs, rfs_config_rf, rfs_config_rf_rays and
    rfs_config_rf_gauss drop the table; rfs_config_swd, rfs_config_swd_modes and the other three table
    setters (successful or failed) keep it; a failed rfs_config_swd* or rfs_config_rf* keeps it; which = 2
    ignores it."""
    cfg = f1_config()
    nt = cfg["nt"]
    X, sets = _rows(B=96, seed=10)
    c = Context(0)
    try:
        _configure(c, 0)
        dobs = _stations(c, 0, G1)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        plain = c.misfit_grad_host(X, 0, sets=sets)
        c.config_obs_gauss(G1)
        table = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(table[0], plain[0])
        # which = 2 ignores the table
        c.config_obs(dobs[:, nt:], SIGMA1, SIGMA2)
        swd_plain = c.misfit_grad_host(X, 2, sets=sets)
        c.config_obs_gauss(G1)
        _assert_same(c.misfit_grad_host(X, 2, sets=sets), swd_plain, "which = 2 ignores the table")
        c.config_obs(dobs, SIGMA1, SIGMA2)
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "config_obs_sets drops")
        c.config_obs_gauss(G1)
        # kept: the SWD configuration and the other setters, with tables of the shared values (the bits of none)
        c.config_swd(7, T, T.copy())
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "config_swd keeps")
        modes = np.zeros(1, dtype=np.int32)
        assert c.L.rfs_config_swd_modes(c.h, 7, T.size, T.ctypes.data_as(_dp), T.size, T.ctypes.data_as(_dp),
                                        0, None, 0, None, 1, modes.ctypes.data_as(ctypes.POINTER(ctypes.c_int)),
                                        0, 1) == 0
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "config_swd_modes keeps")
        c.config_obs_rays(np.full(S, cfg["ray_p"]))
        c.config_obs_periods(np.ones((S, 2 * T.size), dtype=bool))
        c.config_obs_rf_samples(np.ones((S, nt), dtype=bool))
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "other setters keep")
        for bad in (lambda: c.config_obs_rays(np.full(S, np.nan)),
                    lambda: c.config_obs_periods(np.zeros((S, 2 * T.size), dtype=bool)),
                    lambda: c.config_obs_rf_samples(np.zeros((S, nt), dtype=bool))):
            with pytest.raises(RfsError):
                bad()
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "failed other setters keep")
        # a failed configuration keeps it
        t = np.ascontiguousarray(T[::-1])
        assert c.L.rfs_config_swd(c.h, 7, t.size, t.ctypes.data_as(_dp), t.size, t.ctypes.data_as(_dp), 0, None,
                                  0, None, 0, 0, 1) == RFS_E_ARG
        r = np.array([0.05, 0.06])
        assert c.L.rfs_config_rf_rays(c.h, 7, r.size, r.ctypes.data_as(_dp), 2 * nt, cfg["dt"], cfg["gauss"],
                                      cfg["time_shift"], cfg["water"], 3, 1) == RFS_E_ARG
        g = np.array([1.0, np.nan])
        assert c.L.rfs_config_rf_gauss(c.h, 7, r.size, r.ctypes.data_as(_dp), g.size, g.ctypes.data_as(_dp), nt,
                                       cfg["dt"], cfg["time_shift"], cfg["water"], 1, 1) == RFS_E_ARG
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "failed config_swd / config_rf keep")
        # dropped by every successful rfs_config_rf*
        _configure(c, 1)  # rfs_config_rf_rays
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "config_rf_rays drops")
        c.config_obs_gauss(G1)
        assert c.L.rfs_config_rf(c.h, 7, ctypes.c_double(cfg["ray_p"]), nt, cfg["dt"], cfg["gauss"],
                                 cfg["time_shift"], cfg["water"], 1, 1) == 0
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "config_rf drops")
        c.config_obs_gauss(G1)
        c.config_rf(7, cfg["ray_p"], nt, cfg["dt"], [cfg["gauss"]], cfg["time_shift"], cfg["water"])
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "config_rf_gauss drops")
        # rfs_config_obs (the one-set call)
        r3 = sets == 3
        c.config_obs(dobs[3], SIGMA1[3], SIGMA2[3])
        want = c.misfit_grad_host(X[r3], 0)
        c.config_obs_gauss(G1[3:4])
        assert np.array_equal(c.misfit_grad_host(X[r3], 0)[0], table[0][r3])
        d3 = np.ascontiguousarray(dobs[3])
        assert c.L.rfs_config_obs(c.h, SIGMA1[3], SIGMA2[3], d3.ctypes.data_as(_dp), d3.size) == 0
        _assert_same(c.misfit_grad_host(X[r3], 0), want, "config_obs drops")
    finally:
        c.close()


def _boxes(nsta):
    b = np.repeat(driver_bounds(f1_true_model())[None], nsta, axis=0)
    for s in range(nsta):
        b[s, :7, 0] *= 1.0 + 0.04 * s
        b[s, :7, 1] *= 1.0 - 0.03 * s
    return b


@pytest.mark.parametrize("sampler", [0, 1])
def test_hmc_over_stations_with_widths_equals_single_station_runs(sampler):
    nsta, K = 3, 6
    kw = (dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=6, ndraws=1, max_iters=14) if sampler == 0 else
          dict(dt=0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=3, ndraws=3, max_iters=14))
    kw.update(want_samples=True, log_accepts=kw["max_iters"])
    boxes = _boxes(nsta)
    gauss = [1.0, 2.5]
    c = Context(0)
    try:
        _configure(c, 0, gauss=gauss)
        dobs = _stations(c, 0, G2, nsta, seed=5)
    finally:
        c.close()
    want = {}
    for s in range(nsta):
        c = Context(0)
        try:
            _configure(c, 0, gauss=G2[s].tolist())
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
            want[s] = c.hmc_run(sampler, np.arange(K), boxes[s], **kw)
        finally:
            c.close()
    c = Context(0)
    try:
        _configure(c, 0, gauss=gauss)
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        c.config_obs_gauss(G2[:nsta])
        ids = np.tile(np.arange(K), nsta)
        sets = np.repeat(np.arange(nsta), K)
        for resident in (0, 5):
            c.set_hmc_options(resident=resident)
            got = c.hmc_run(sampler, ids, boxes, sets=sets, **kw)
            assert len(set(got["n_iter"].tolist())) > 1  # chains finish at different steps: compaction
            for s in range(nsta):
                r = sets == s
                for k in ("samples", "misfit", "n_iter", "n_acc", "accept_seq", "initmodel", "dt"):
                    assert np.array_equal(got[k][r], want[s][k], equal_nan=True), (resident, s, k)
    finally:
        c.set_hmc_options(resident=0)
        c.close()


def _f1_joint(gauss):
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    cfg = f1_config()
    rf = ReceiverFunc(cfg["ray_p"], cfg["nt"], cfg["dt"], gauss, cfg["time_shift"], cfg["water"],
                      cfg["rf_type"], cfg["method"])
    return Joint_RF_SWD(1.0, 1.0, rf, SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"]))


def test_station_array_with_widths_matches_its_station_models(tmp_path):
    from rfsurfhmc_b200.model.stations import StationArray
    from rfsurfhmc_b200.pyhmc.hmc import HamitonianMC
    gauss = [1.0, 2.5]
    c = Context(0)
    try:
        _configure(c, 0, gauss=gauss)
        dobs = _stations(c, 0, G2, 3, seed=6)
    finally:
        c.close()
    nt = f1_config()["nt"]
    use = np.ones((3, 1, 2, nt), dtype=bool)
    use[2, :, 0] = False  # station 2 fits its second width only
    sa = StationArray(_f1_joint(gauss), dobs, sigma1=[1.0, 0.5, 2.0], names=["AA01", "BB02", "CC03"],
                      rf_use=use, gauss=G2[:3])
    X, _ = _rows(B=18, seed=2, nsta=3)
    got = sa.misfit_and_grad_batch(X, np.arange(18) % 3)
    for s in range(3):
        m = sa.station_model(s)
        assert m.rfmodel.gauss == (G2[s].tolist() if s < 2 else [G2[2, 1]])
        rows = [v[s::3] for v in got]
        if s == 2:  # the single-station model's synthetics hold its fitted width only
            rows[2] = rows[2][:, nt:]
        for k, (u, v) in enumerate(zip(rows, m.misfit_and_grad_batch(X[s::3]))):
            assert np.array_equal(u, v, equal_nan=True), (s, k)
    bounds = driver_bounds(f1_true_model())
    hmc = HamitonianMC(sa, bounds, 0.1, (5, 20), 3, 991206, 4, 1, name="ch", outdir=str(tmp_path))
    hmc.max_iters = 12
    out = hmc.sample_chains([0, 1, 0], stations=[0, 0, 1], save=True)
    one = HamitonianMC(sa.station_model(1), bounds, 0.1, (5, 20), 3, 991206, 4, 1, name="one",
                       outdir=str(tmp_path))
    one.max_iters = 12
    ref = one.sample_chains([0])
    for k in ("misfit", "samples", "n_iter", "n_acc"):
        assert np.array_equal(out[k][2], ref[k][0], equal_nan=True), k
    assert np.array_equal(np.load(tmp_path / "BB02" / "ch.0.npz")["obs"], dobs[1])


def test_driver_runs_a_stations_file_with_widths(tmp_path):
    from rfsurfhmc_b200 import driver
    with open(os.path.join(ROOT, "tests", "golden", "f1_param.yaml")) as fh:
        param = yaml.safe_load(fh)
    g = param["rf"]["gauss"]
    c = Context(0)
    try:
        _configure(c, 0, rays=param["rf"]["ray_p"], gauss=g)
        dobs = _stations(c, 0, G1[2:], 2, seed=7)
    finally:
        c.close()

    def run(tag, **keys):
        param["hmc"].update(OUTPUT_DIR=str(tmp_path / tag), nsamples=3, ndraws=1)
        path = tmp_path / f"{tag}.npz"
        np.savez(path, **keys)
        return driver.run(param, "base", 2, save_chains=False, max_iters=8, stations=str(path))[0]

    both = run("both", dobs=dobs, names=np.array(["N1", "N2"]), gauss=G1[2:4])
    alone = run("alone", dobs=dobs[1:], names=np.array(["N2"]), gauss=G1[3:4])
    shared = run("shared", dobs=dobs, names=np.array(["N1", "N2"]))
    assert np.array_equal(np.load(tmp_path / "both" / "N2" / "misfit.npy"), both[2:], equal_nan=True)
    assert np.array_equal(both[2:], alone, equal_nan=True)
    assert not np.array_equal(both[2:], shared[2:], equal_nan=True)


def test_joint_evaluator_with_obs_gauss():
    from rfsurfhmc_b200.batched import JointEvaluator
    cfg = f1_config()
    cfg.update(sigma1=SIGMA1, sigma2=SIGMA2, gauss=[1.0, 2.5])
    c = Context(0)
    try:
        _configure(c, 0, gauss=cfg["gauss"])
        dobs = _stations(c, 0, G2)
        X, sets = _rows(B=128, seed=12)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_gauss(G2)
        want = c.misfit_grad_host(X, 0, sets=sets)
    finally:
        c.close()
    ev = JointEvaluator(cfg, dobs, 7, obs_gauss=G2)
    dev = torch.device("cuda", 0)
    U, G, D, F = ev(torch.from_numpy(X).to(dev), torch.from_numpy(sets).to(dev))
    torch.cuda.synchronize(dev)
    got = [U.cpu().numpy(), G.cpu().numpy(), D.cpu().numpy(), F.cpu().numpy().astype(bool)]
    ev.ctx.close()
    _assert_same(got, want, "JointEvaluator")
