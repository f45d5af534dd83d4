"""Receiver functions at several Gaussian widths in one objective (rfs_config_rf_gauss): every trace of
a width list must be the trace of a one-width configuration, misfit and gradient the sums over the
(ray, width) passes, and the station tables, the HMC and the Python classes must take the [ray][gauss][nt]
data layout."""
import ctypes
import os
import numpy as np
import pytest
import torch
import yaml
from oracle import hmc_ref
from rfsurfhmc_b200._lib import Context, RfsError
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RFS_E_ARG = -2
CFG = f1_config()
NT = CFG["nt"]
NSW = 2 * len(CFG["tRc"])
WIDTHS = [1.0, 2.5, 5.0]
RAYS_P = [0.04, 0.055, 0.07]
RAYS_S = [0.1, 0.11, 0.12]  # S-wave RF: slowness of teleseismic S
METHODS = ["freq", "time"]


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _configure(c, which, method="freq", rf_type="P", rays=0.045, gauss=WIDTHS[:2], n=7, nt=NT, dt=None):
    if which != 1:
        c.config_swd(n, tRc=CFG["tRc"], tRg=CFG["tRg"])
    if which != 2:
        c.config_rf(n, rays, nt, CFG["dt"] if dt is None else dt, gauss, CFG["time_shift"], CFG["water"], rf_type,
                    method)


def _rows(B=240, seed=8, nsta=1):
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


def _observed(c, which, nsta=1, seed=3, table=None):
    """Synthetics of seeded perturbations of the F1 true model plus seeded noise, from the configured c."""
    c.config_obs(np.zeros((nsta, c.ndata(which))))
    if table is not None:
        c.config_obs_rays(table)
    Xs = perturbed_models(f1_true_model(), nsta, seed=seed, rel=0.05)
    _, _, d, _ = c.misfit_grad_host(Xs, which, sets=np.arange(nsta))
    d = np.where(np.isfinite(d), d, 0.0)
    return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)


def _passes(method, rf_type, rays, widths, dobs_rf, X, n=7, nt=NT, dt=None):
    """Reference: one one-ray, one-width context per (ray, width) pass, summed on the host in pass order
    [ray][gauss].  Returns U, grad and the traces [B][nray][G][nt]."""
    rays = list(np.atleast_1d(rays))
    U = np.zeros(len(X))
    g = np.zeros(X.shape)
    d = np.zeros((len(X), len(rays), len(widths), nt))
    c = Context(0)
    try:
        for ir, p in enumerate(rays):
            for ig, a in enumerate(widths):
                _configure(c, 1, method, rf_type, float(p), float(a), n=n, nt=nt, dt=dt)
                o = (ir * len(widths) + ig) * nt
                c.config_obs(dobs_rf[o:o + nt])
                Ui, gi, di, fi = c.misfit_grad_host(X, 1)
                assert fi.all()
                if ir == 0 and ig == 0:
                    U, g = Ui, gi
                else:
                    U, g = U + Ui, g + gi
                d[:, ir, ig] = di
    finally:
        c.close()
    return U, g, d


def _check_against_passes(got, want, method, tag):
    U, g, d = want
    assert np.array_equal(got[2][:, :d[0].size], d.reshape(len(d), -1)), (tag, "dsyn")
    if method == "time":
        assert np.array_equal(got[0], U), (tag, "U")
        assert np.array_equal(got[1], g), (tag, "grad")
    else:
        assert np.all(np.abs(got[0] - U) <= 1e-12 * np.abs(U)), (tag, "U")
        assert np.all(np.abs(got[1] - g) <= 1e-10 * np.abs(g).max(axis=1, keepdims=True)), (tag, "grad")


CASES = [(m, t, nr, G) for m in METHODS for t in ("P", "S") for nr in (1, 3) for G in (2, 3)]


@pytest.mark.parametrize("method,rf_type,nray,G", CASES, ids=[f"{m}-{t}-r{nr}-g{G}" for m, t, nr, G in CASES])
def test_widths_equal_one_width_passes(method, rf_type, nray, G):
    rays = (RAYS_P if rf_type == "P" else RAYS_S)[:nray]
    widths = WIDTHS[:G]
    X, _ = _rows(B=160, seed=10 + nray + G)
    n1 = nray * G * NT
    c = Context(0)
    try:
        _configure(c, 0, method, rf_type, rays, widths)
        assert c.ndata(0) == n1 + NSW and c.ngauss == G
        dobs = _observed(c, 0)[0]
        c.config_obs(dobs)
        joint = c.misfit_grad_host(X, 0)
        c.config_obs(dobs[:n1])
        rf = c.misfit_grad_host(X, 1)
        c.config_obs(dobs[n1:])
        sw = c.misfit_grad_host(X, 2)
    finally:
        c.close()
    assert rf[3].all()
    _check_against_passes(rf, _passes(method, rf_type, rays, widths, dobs[:n1], X), method, "rf")
    # joint: RF + wt SWD with the joint weight of n1 = nray G nt RF samples
    ok = joint[3]
    assert np.array_equal(ok, sw[3]) and ok.sum() > len(X) // 2 and not ok.all()
    wt = (CFG["sigma1"] / CFG["sigma2"]) ** 2 * n1 / NSW
    U = rf[0][ok] + wt * sw[0][ok]
    g = rf[1][ok] + wt * sw[1][ok]
    assert np.all(np.abs(joint[0][ok] - U) <= 1e-12 * np.abs(U))
    assert np.all(np.abs(joint[1][ok] - g) <= 1e-12 * np.abs(g).max(axis=1, keepdims=True))
    assert np.array_equal(joint[2][ok][:, :n1], rf[2][ok])
    assert np.array_equal(joint[2][~ok], np.broadcast_to(dobs, joint[2][~ok].shape))


def test_widths_against_the_oracle_at_c3_sizes(oracle):
    """n = 40, nt = 2048, three ray parameters and three widths against oracle.joint_batch per pass, at
    the tolerances of test_gpu_sizes.py."""
    from test_gpu_sizes import TOL_RF, TOL_G, NTH, layered, rel, grad_err
    n, B, nt, dt = 40, 16, 2048, 0.05
    X = layered(B, n, 22)
    rays = (0.04, 0.06, 0.08)
    base = dict(f1_config(), nt=nt, dt=dt, time_shift=5.0, water=1e-3)
    dobs = 0.02 * np.random.default_rng(1).standard_normal(len(rays) * len(WIDTHS) * nt)
    c = Context(0)
    try:
        c.config_rf(n, list(rays), nt, dt, WIDTHS, 5.0, 1e-3, "P", "freq")
        c.config_obs(dobs)
        U, g, d, f = c.misfit_grad_host(X, which=1)
    finally:
        c.close()
    assert d.shape == (B, 9 * nt) and f.all()
    Us, gs = 0.0, 0.0
    for ir, p in enumerate(rays):
        for ig, a in enumerate(WIDTHS):
            o = (ir * len(WIDTHS) + ig) * nt
            Ua, ga, da, fa = oracle.joint_batch(X, dobs[o:o + nt], dict(base, ray_p=p, gauss=a), which=1, nthreads=NTH)
            assert np.max(np.abs(d[:, o:o + nt] - da)) <= TOL_RF * np.max(np.abs(da)), (p, a)
            Us, gs = Us + Ua, gs + ga
    assert rel(U, Us) <= 1e-8 and grad_err(g, gs).max() <= TOL_G


def test_nt_4096_with_three_widths():
    """The largest shared-memory case of rf_decon_kernel (nft = 4096 with the weight accumulator)."""
    n, nt, dt = 40, 4096, 0.025
    from test_gpu_sizes import layered
    X = layered(8, n, 5)
    dobs = 0.02 * np.random.default_rng(2).standard_normal(3 * nt)
    c = Context(0)
    try:
        c.config_rf(n, 0.06, nt, dt, WIDTHS, CFG["time_shift"], CFG["water"], "P", "freq")
        c.config_obs(dobs)
        got = c.misfit_grad_host(X, 1)
    finally:
        c.close()
    assert got[3].all() and np.isfinite(got[2]).all()
    _check_against_passes(got, _passes("freq", "P", 0.06, WIDTHS, dobs, X, n=n, nt=nt, dt=dt), "freq", "nt4096")


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("method", METHODS)
def test_one_element_list_gives_the_bits_of_config_rf_rays(which, method):
    X, _ = _rows(B=128, seed=4)
    outs = []
    for gauss in (CFG["gauss"], [CFG["gauss"]]):
        c = Context(0)
        try:
            _configure(c, which, method, rays=RAYS_P[:2], gauss=gauss)
            assert c.ngauss == 1
            dobs = _observed(c, which, seed=9)[0]
            c.config_obs(dobs)
            outs.append(c.misfit_grad_host(X, which))
        finally:
            c.close()
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a, b, equal_nan=True)


# ---- station tables
S = 4
SIGMA1 = np.array([1.0, 0.5, 2.0, 1.0])
SIGMA2 = np.array([1.0, 1.5, 1.0, 0.25])
TABLE = np.array([[0.04, 0.06], [0.045, 0.065], [0.05, 0.07], [0.042, 0.071]])
NR, G2 = 2, 2


def _masks():
    """[S][ray][gauss][nt]: station 0 fits everything, station 1 misses width 1 on every ray, station 2
    misses ray 0, station 3 fits a window of each trace."""
    u = np.ones((S, NR, G2, NT), dtype=bool)
    u[1, :, 1] = False
    u[2, 0] = False
    u[3] = False
    rng = np.random.default_rng(1)
    for r in range(NR):
        for g in range(G2):
            a = int(rng.integers(0, 40))
            u[3, r, g, a:a + 60] = True
    return u


def _grouped(which, method, dobs, X, sets, use=None, ctx=None):
    c = Context(0) if ctx is None else ctx
    try:
        _configure(c, which, method, rays=list(TABLE[0]), gauss=WIDTHS[:G2])
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_rays(TABLE)
        if use is not None:
            c.config_obs_rf_samples(use)
        return c.misfit_grad_host(X, which, sets=sets)
    finally:
        if ctx is None:
            c.close()


def _station_data(which, method):
    c = Context(0)
    try:
        _configure(c, which, method, rays=list(TABLE[0]), gauss=WIDTHS[:G2])
        return _observed(c, which, S, seed=5, table=TABLE)
    finally:
        c.close()


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "freq"), (0, "time"), (1, "time")])
def test_station_tables_with_widths_equal_per_station_contexts(which, method):
    """Stations with a whole width or a whole ray missing equal a one-station context on their observed
    rays and widths; the windowed station equals a one-station context holding its own mask."""
    use = _masks()
    dobs = _station_data(which, method)
    X, sets = _rows(B=200, seed=6, nsta=S)
    got = _grouped(which, method, dobs, X, sets, use.reshape(S, -1))
    nrf = NR * G2 * NT
    for s in range(S):
        r = np.flatnonzero(sets == s)
        obs = use[s].all(axis=2)
        c = Context(0)
        try:
            if s < 3:
                rays, widths = obs.any(axis=1), obs.any(axis=0)
                _configure(c, which, method, rays=list(TABLE[s][rays]), gauss=list(np.asarray(WIDTHS[:G2])[widths]))
                pos = np.flatnonzero(use[s].reshape(-1))
                if which == 0:
                    pos = np.concatenate((pos, nrf + np.arange(NSW)))
                c.config_obs(dobs[s][pos], SIGMA1[s], SIGMA2[s])
            else:
                pos = np.arange(dobs.shape[1])
                _configure(c, which, method, rays=list(TABLE[s]), gauss=WIDTHS[:G2])
                c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
                c.config_obs_rf_samples(use[s].reshape(1, -1))
            U, g, d, f = c.misfit_grad_host(X[r], which)
        finally:
            c.close()
        assert np.array_equal(got[0][r], U) and np.array_equal(got[1][r], g) and np.array_equal(got[3][r], f), s
        assert np.array_equal(got[2][r][:, pos], d, equal_nan=True), s
    if which == 0:
        assert not got[3].all()


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


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "freq"), (1, "time")])
def test_out_of_range_set_fails_only_its_row(which, method):
    use = _masks().reshape(S, -1)
    dobs = _station_data(which, method)
    X, sets = _rows(B=96, seed=4, nsta=S)
    c = Context(0)
    try:
        want = _grouped(which, method, dobs, X, sets, use, ctx=c)
        s = sets.copy()
        bad = np.array([3, 40, 95])
        s[bad] = [-1, S, 1 << 30]
        got = _dev_eval(c, X, s, which)
    finally:
        c.close()
    assert (got[0][bad] == 0).all() and (got[1][bad] == 0).all() and np.isnan(got[2][bad]).all()
    assert not got[3][bad].any()
    keep = np.setdiff1d(np.arange(len(X)), bad)
    for a, b in zip(got[:3], want[:3]):
        assert np.array_equal(a[keep], b[keep], equal_nan=True)
    assert np.array_equal(got[3][keep].astype(bool), want[3][keep])


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "time")])
def test_chunked_batch_with_widths(which, method):
    """A 1 MiB workspace budget forces many 32-row chunks."""
    use = _masks().reshape(S, -1)
    dobs = _station_data(which, method)
    X, sets = _rows(B=300, seed=2, nsta=S)
    want = _grouped(which, method, dobs, X, sets, use)
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
        n0 = c.launches
        got = _grouped(which, method, dobs, X, sets, use, ctx=c)
        assert c.launches - n0 > 40
    finally:
        c.close()
    for a, b in zip(got, want):
        assert np.array_equal(a, b, equal_nan=True)


def _raw_gauss(c, widths, n=7, nray=1, rays=(0.045,)):
    r = np.ascontiguousarray(rays, dtype=np.float64)
    if widths is None:
        return c.L.rfs_config_rf_gauss(c.h, n, nray, _dp(r), 2, None, NT, CFG["dt"], CFG["time_shift"],
                                       CFG["water"], 1, 1)
    w = np.ascontiguousarray(widths, dtype=np.float64)
    return c.L.rfs_config_rf_gauss(c.h, n, nray, _dp(r), w.size, _dp(w), NT, CFG["dt"], CFG["time_shift"],
                                   CFG["water"], 1, 1)


def test_config_rf_gauss_errors_and_table_lifetime():
    dobs = _station_data(0, "freq")
    X, sets = _rows(B=96, seed=3, nsta=S)
    use = _masks().reshape(S, -1)
    c = Context(0)
    try:
        _configure(c, 0, rays=list(TABLE[0]), gauss=WIDTHS[:G2])
        c.config_obs(dobs, SIGMA1, SIGMA2)
        plain = c.misfit_grad_host(X, 0, sets=sets)
        c.config_obs_rays(TABLE)
        c.config_obs_rf_samples(use)
        c.config_obs_periods(np.tile(np.arange(NSW) % 3 != 0, (S, 1)))
        tabled = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(tabled[0], plain[0])
        # bad lists: RFS_E_ARG, and the context (configuration and all three tables) is unchanged
        for bad in ([], list(np.linspace(1, 2, 17)), [1.0, np.nan], [1.0, np.inf], [2.5, 0.0], [-1.0, 1.0], None):
            assert _raw_gauss(c, bad, nray=2, rays=TABLE[0]) == RFS_E_ARG, bad
        assert _raw_gauss(c, [1.0, 2.0], n=1, nray=2, rays=TABLE[0]) == RFS_E_ARG  # a bad layer count
        for a, b in zip(c.misfit_grad_host(X, 0, sets=sets), tabled):
            assert np.array_equal(a, b, equal_nan=True)
        # nrf is checked against nray G nt
        with pytest.raises(RfsError) as e:
            c.config_obs_rf_samples(use.reshape(S, NR, G2, NT)[:, :, 0])
        assert e.value.code == RFS_E_ARG
        # a successful call drops the ray and RF-sample tables and keeps the period table
        c.config_obs_periods(np.tile(np.arange(NSW) % 3 != 0, (S, 1)))
        periods_only = Context(0)
        try:
            _configure(periods_only, 0, rays=list(TABLE[0]), gauss=WIDTHS[:G2])
            periods_only.config_obs(dobs, SIGMA1, SIGMA2)
            periods_only.config_obs_periods(np.tile(np.arange(NSW) % 3 != 0, (S, 1)))
            want = periods_only.misfit_grad_host(X, 0, sets=sets)
        finally:
            periods_only.close()
        assert _raw_gauss(c, WIDTHS[:G2], nray=2, rays=TABLE[0]) == 0
        for a, b in zip(c.misfit_grad_host(X, 0, sets=sets), want):
            assert np.array_equal(a, b, equal_nan=True)
    finally:
        c.close()
    # rfs_config_rf and rfs_config_rf_rays still accept their one width unchecked, as before
    c = Context(0)
    try:
        r = np.array([0.045])
        assert c.L.rfs_config_rf_rays(c.h, 7, 1, _dp(r), NT, CFG["dt"], 0.0, CFG["time_shift"], CFG["water"], 1, 1) == 0
        assert c.L.rfs_config_rf(c.h, 7, ctypes.c_double(0.045), NT, CFG["dt"], -1.0, CFG["time_shift"],
                                 CFG["water"], 1, 1) == 0
    finally:
        c.close()


# ---- HMC
def _hmc_kw(sampler):
    kw = (dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=6, ndraws=1, max_iters=14) if sampler == 0 else
          dict(dt=0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=3, ndraws=3, max_iters=14))
    kw.update(want_samples=True, want_syn=True, log_accepts=kw["max_iters"])
    return kw


def _oracle_two_width_f(O, dobs, widths):
    """The joint objective over the widths, composed from the oracle's one-width RF objectives and its SWD
    objective, with the joint weight of n1 = G nt RF samples."""
    n1 = len(widths) * NT
    wt = (CFG["sigma1"] / CFG["sigma2"]) ** 2 * n1 / NSW

    def f(x):
        x = np.asarray(x)[None, :]
        Us, gs, ds = 0.0, 0.0, []
        for ig, a in enumerate(widths):
            U, g, d, _ = O.joint_batch(x, dobs[ig * NT:(ig + 1) * NT], dict(CFG, gauss=a), which=1)
            Us, gs = Us + U[0], gs + g[0]
            ds.append(d[0])
        U, g, d, fl = O.joint_batch(x, dobs[n1:], CFG, which=2)
        if not fl[0]:
            return 0.0, np.zeros(x.shape[1]), dobs, False
        return float(Us + wt * U[0]), gs + wt * g[0], np.concatenate(ds + [d[0]]), True
    return f


def test_hmc_accept_sequences_against_the_oracle_sampler(oracle):
    widths = WIDTHS[:2]
    bounds = driver_bounds(f1_true_model())
    c = Context(0)
    try:
        _configure(c, 0, gauss=widths)
        dobs = _observed(c, 0, seed=4)[0]
        c.config_obs(dobs)
        f = _oracle_two_width_f(oracle, dobs, widths)
        niter = 12
        out = c.hmc_run(0, [0, 1, 2], bounds, 0.1, Lrange=(5, 20), seed=991206, nsamples=40, ndraws=5,
                        max_iters=niter, want_samples=True, log_accepts=niter)
        for i, cid in enumerate([0, 1, 2]):
            R = hmc_ref.run_base(f, bounds, 0.1, (5, 20), 991206 + cid, nsamples=40, ndraws=5, max_iters=niter)
            assert np.allclose(out["initmodel"][i], R.initmodel, rtol=0, atol=1e-14)
            assert list(out["accept_seq"][i][:out["n_iter"][i]]) == R.accepts, cid
            assert out["n_acc"][i] == R.n_acc
        niter = 8
        out = c.hmc_run(1, [0, 5], bounds, 0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=20, ndraws=4,
                        max_iters=niter, want_samples=True, log_accepts=niter)
        for i, cid in enumerate([0, 5]):
            R = hmc_ref.run_da(f, bounds, 0.02, 10, 0.65, 991206 + cid, nsamples=20, ndraws=4, max_iters=niter)
            assert list(out["accept_seq"][i][:out["n_iter"][i]]) == R.accepts, cid
            assert np.isclose(out["dt"][i], R.dt, rtol=1e-6)
    finally:
        c.close()


@pytest.mark.parametrize("sampler", [0, 1])
def test_grouped_hmc_with_widths_equals_single_station_runs(sampler):
    nsta, K = 3, 5
    kw = _hmc_kw(sampler)
    bounds = driver_bounds(f1_true_model())
    dobs = _station_data(0, "freq")[:nsta]
    want = []
    for s in range(nsta):
        c = Context(0)
        try:
            _configure(c, 0, rays=list(TABLE[s]), gauss=WIDTHS[:G2])
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
            want.append(c.hmc_run(sampler, np.arange(K), bounds, **kw))
        finally:
            c.close()
    c = Context(0)
    try:
        _configure(c, 0, rays=list(TABLE[0]), gauss=WIDTHS[:G2])
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        c.config_obs_rays(TABLE[:nsta])
        sets = np.repeat(np.arange(nsta), K)
        got = c.hmc_run(sampler, np.tile(np.arange(K), nsta), bounds, sets=sets, **kw)
    finally:
        c.close()
    for s in range(nsta):
        r = sets == s
        for k in ("samples", "misfit", "n_iter", "n_acc", "accept_seq", "initmodel", "dt", "syn"):
            assert np.array_equal(got[k][r], want[s][k], equal_nan=True), (s, k)


# ---- Python end to end
def _rf_model(gauss, rays=0.045, method="freq"):
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    return ReceiverFunc(rays, NT, CFG["dt"], gauss, CFG["time_shift"], CFG["water"], CFG["rf_type"], method)


@pytest.mark.parametrize("method", METHODS)
def test_receiver_func_with_widths_sums_its_one_width_objects(method):
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    from rfsurfhmc_b200.model.model_surf import SurfWD
    rays = RAYS_P[:2]
    m = _rf_model(WIDTHS, rays, method)
    assert m.nt == 2 * 3 * NT and m.nt_trace == NT and m.ngauss == 3
    x0 = f1_true_model()
    x = x0 * 1.03
    dobs = m.forward(x0)
    assert dobs.shape == (m.nt,)
    m.set_obsdata(dobs)
    U, g, d = m.misfit_and_grad(x)
    # forward() (the librf drop-in per trace, in [ray][gauss] order) against the fused objective's traces;
    # the time method's drop-in forward runs the propagator with the reference's float pi, the objective
    # with the double one, and deconit's spike picking may then differ
    if method == "freq":
        assert np.max(np.abs(m.forward(x) - d)) <= 1e-10 * np.max(np.abs(d))
    else:
        assert m.forward(x).shape == d.shape
    Us, gs = 0.0, 0.0
    d3 = dobs.reshape(2, 3, NT)
    for ig, a in enumerate(WIDTHS):
        one = _rf_model(a, rays, method)
        one.set_obsdata(d3[:, ig].reshape(-1))
        Ui, gi, di = one.misfit_and_grad(x)
        assert np.array_equal(di.reshape(2, NT), d.reshape(2, 3, NT)[:, ig])
        Us, gs = Us + Ui, gs + gi
    assert abs(U - Us) <= 1e-12 * abs(Us) and np.max(np.abs(g - gs)) <= 1e-10 * np.max(np.abs(gs))
    # Joint_RF_SWD on top, through rfmodel.nt
    swd = SurfWD(tRc=CFG["tRc"], tRg=CFG["tRg"])
    j = Joint_RF_SWD(1.0, 1.0, m, swd)
    assert j.ndata == m.nt + NSW
    j.set_obsdata(dobs, swd.forward(x0)[0])
    Uj, gj, dj, fj = j.misfit_and_grad(x)
    assert fj and np.array_equal(dj[:m.nt], d)
    c = Context(0)
    try:
        _configure(c, 0, method, rays=rays, gauss=WIDTHS)
        c.config_obs(j.dobs)
        U2, g2, d2, f2 = c.misfit_grad_host(x[None, :], 0)
    finally:
        c.close()
    assert Uj == U2[0] and np.array_equal(gj, g2[0]) and np.array_equal(dj, d2[0])


def test_station_array_with_widths_matches_its_station_models():
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.stations import StationArray
    use = _masks()[:3]
    dobs = _station_data(0, "freq")[:3]
    t = Joint_RF_SWD(1.0, 1.0, _rf_model(WIDTHS[:G2], list(TABLE[0])), SurfWD(tRc=CFG["tRc"], tRg=CFG["tRg"]))
    sa = StationArray(t, dobs, sigma1=SIGMA1[:3], sigma2=SIGMA2[:3], ray_p=TABLE[:3], rf_use=use)
    X, _ = _rows(B=18, seed=2)
    st = np.arange(18) % 3
    got = sa.misfit_and_grad_batch(X, st)
    for s in range(3):
        m = sa.station_model(s)
        b = m.misfit_and_grad_batch(X[st == s])
        for i in (0, 1, 3):
            assert np.array_equal(got[i][st == s], b[i]), s
    assert sa.station_model(1).rfmodel.gauss == [WIDTHS[0]] and sa.station_model(2).rfmodel.nray == 1


def test_driver_runs_a_width_list_and_a_stations_file_with_4d_rf_use(tmp_path):
    from rfsurfhmc_b200 import driver
    with open(os.path.join(ROOT, "tests", "golden", "f1_param.yaml")) as fh:
        param = yaml.safe_load(fh)
    param["rf"]["gauss"] = [1.0, 2.5]
    param["hmc"].update(OUTPUT_DIR=str(tmp_path / "synth"), nsamples=3, ndraws=1)
    misfit, n_iter, _ = driver.run(param, "base", 2, save_chains=True, max_iters=6)
    assert misfit.shape == (2, 3) and np.load(tmp_path / "synth" / "real_syn.npy").shape == (2 * NT + NSW,)
    c = Context(0)
    try:
        _configure(c, 0, gauss=[1.0, 2.5])
        dobs = _observed(c, 0, nsta=2, seed=7)
    finally:
        c.close()
    use = np.ones((2, 1, 2, NT), dtype=bool)
    use[0, 0, 1] = False
    use[1, 0, :, 60:] = False

    def run(tag, **keys):
        param["hmc"].update(OUTPUT_DIR=str(tmp_path / tag), nsamples=3, ndraws=1)
        path = tmp_path / f"{tag}.npz"
        np.savez(path, **keys)
        return driver.run(param, "base", 2, save_chains=True, max_iters=8, stations=str(path))[0]

    both = run("both", dobs=dobs, names=np.array(["N1", "N2"]), rf_use=use)
    alone = run("alone", dobs=dobs[1:], names=np.array(["N2"]), rf_use=use[1:].reshape(1, -1))
    assert np.array_equal(np.load(tmp_path / "both" / "N2" / "misfit.npy"), both[2:], equal_nan=True)
    assert np.array_equal(both[2:], alone, equal_nan=True)
