"""[vs, thk, vpvs] parameterisation on the device (rfs_config_param RFS_PARAM_VS_THK_VPVS): U, dsyn and the
three gradient blocks against the reference composed from the oracle's per-field kernels
(tests/vpvs_ref.py: vpvs_objective), identity with the Brocher path at k = vp_B(vs)/vs, central
differences in k, grouped evaluations with every per-set table, and the device HMC against the samplers'
restatement.  Tolerances are the Brocher-path ones of test_gpu_parity.py: c <= 1e-6 relative, RF <= 1e-5 of
the trace peak, gradients <= 1e-4 of the largest component of that gradient block."""
import numpy as np
import pytest
import vpvs_ref
from oracle.oracle import brocher
from rfsurfhmc_b200._lib import Context
from rfsurfhmc_b200.fixtures import (f1_config, f1_true_model, driver_bounds_vpvs, sorted_uniform_models_vpvs)

pytestmark = pytest.mark.gpu
TOL_C, TOL_RF, TOL_G = 1e-6, 1e-5, 1e-4


@pytest.fixture(autouse=True)
def default_param_after(ctx):
    """the session context goes back to the default [vs, thk] layout for the other test modules"""
    yield
    ctx.config_param(False)


def x3(x2, scale=1.02):
    """[vs, thk] -> [vs, thk, k] with k near Brocher's vp/vs of each layer."""
    n = x2.size // 2
    vs = x2[:n]
    return np.hstack((x2, brocher(vs)[0] / vs * scale))


def models(x, B, seed):
    X = sorted_uniform_models_vpvs(driver_bounds_vpvs(x), B, seed)
    rng = np.random.default_rng(seed + 1)
    P = x * (1 + 0.05 * rng.uniform(-1, 1, (B, x.size)))
    P[:, (x.size // 3) * 2 - 1] = rng.uniform(0, 2, B)
    return np.vstack((X, P))


def configure(c, n, cfg, which, vpvs=True):
    c.config_param(vpvs)
    if which != 1:
        c.config_swd(n, cfg.get("tRc"), cfg.get("tRg"), cfg.get("tLc"), cfg.get("tLg"), mode=cfg.get("mode", 0),
                     sphere=cfg.get("sphere", False))
    if which != 2:
        c.config_rf(n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                    cfg["rf_type"], cfg["method"])


def nrf(cfg):
    return cfg["nt"] * np.size(cfg["ray_p"]) * np.size(cfg["gauss"])


def data_of(cfg, which):
    sl = slice(0, None) if which == 0 else (slice(0, nrf(cfg)) if which == 1 else slice(nrf(cfg), None))
    return sl


def check_parity(ctx, oracle, cfg, X, dobs, which, min_ok=0.99, gmax=1e-2):
    n = X.shape[1] // 3
    sl = data_of(cfg, which)
    configure(ctx, n, cfg, which)
    ctx.config_obs(dobs[sl])
    U1, g1, d1, f1 = ctx.misfit_grad_host(X, which=which)
    assert g1.shape == X.shape
    ref = [vpvs_ref.vpvs_objective(oracle, x, dobs[sl], cfg, which) for x in X]
    f0 = np.array([r[3] for r in ref])
    assert np.array_equal(f0, f1)
    assert f0.sum() >= len(X) // 2
    assert np.all(g1[~f1] == 0.0) and np.all(U1[~f1] == 0.0)
    n1 = nrf(cfg) if which != 2 else 0
    e_u, e_g, e_rf, e_c = [], [], [], []
    for b in np.nonzero(f0)[0]:
        U0, g0, d0, _ = ref[b]
        # a higher mode that does not exist at a period (NaN or 0 in the synthetics) has no kernels: such rows
        # are compared for that pattern only
        missing0 = ~np.isfinite(d0) | (d0 == 0.0)
        assert np.array_equal(~np.isfinite(d1[b]) | (d1[b] == 0.0), missing0), b
        if missing0.any():
            continue
        e_u.append(abs(U1[b] - U0) / max(U0, 1e-12))
        e_g.append(max(np.max(np.abs(g1[b, j * n:(j + 1) * n] - g0[j * n:(j + 1) * n])) /
                       np.max(np.abs(g0[j * n:(j + 1) * n])) for j in range(3)))
        if n1:
            e_rf.append(np.max(np.abs(d1[b, :n1] - d0[:n1])) / np.max(np.abs(d0[:n1])))
        if which != 1:
            e_c.append(np.max(np.abs(d1[b, n1:] - d0[n1:]) / np.abs(d0[n1:])))
    assert len(e_u) >= len(X) // 3
    e_u, e_g = np.array(e_u), np.array(e_g)
    if e_rf:
        assert max(e_rf) <= TOL_RF
    if e_c:
        e_c = np.array(e_c)
        assert np.mean(e_c <= TOL_C) >= min_ok and e_c.max() < 1e-3
    # the root search is chaotic at the 1e-16 level for a few strongly inverted models (DESIGN.md)
    assert np.mean(e_g <= TOL_G) >= min_ok and e_g.max() < gmax, (np.sort(e_g)[-5:])
    assert np.mean(e_u <= 1e-5) >= min_ok


@pytest.mark.parametrize("which", [0, 1, 2])
def test_f1_parity_with_the_oracle_composition(ctx, oracle, which):
    cfg = f1_config()
    x = x3(f1_true_model())
    dobs = vpvs_ref.vpvs_objective(oracle, x, np.zeros(125 + 72), cfg, 0)[2]
    check_parity(ctx, oracle, cfg, models(x, 24, seed=5), dobs, which)


@pytest.mark.parametrize("method,rf_type", [("freq", "S"), ("time", "P"), ("time", "S")])
def test_rf_methods_and_types_parity(ctx, oracle, method, rf_type):
    cfg = dict(f1_config(), method=method, rf_type=rf_type, ray_p=[0.045, 0.07], gauss=[1.5, 3.0])
    x = x3(f1_true_model())
    dobs = vpvs_ref.vpvs_objective(oracle, x, np.zeros(4 * 125), cfg, 1)[2]
    # the time method's argmax spike picking can flip on near-ties (test_gpu_parity.py)
    min_ok, gmax = (0.9, 5e-2) if method == "time" else (0.99, 1e-2)
    check_parity(ctx, oracle, cfg, models(x, 12, seed=7), dobs, 1, min_ok=min_ok, gmax=gmax)


@pytest.mark.parametrize("which", [0, 1, 2])
def test_sphere_love_modes_rays_widths_parity(ctx, oracle, which):
    T = np.arange(3., 13.)  # the first higher mode exists at every period for these models
    cfg = dict(f1_config(), tRc=T, tRg=T.copy(), tLc=T.copy(), tLg=[], mode=[0, 1], sphere=True,
               ray_p=[0.04, 0.065], gauss=[1.0, 2.5])
    x = x3(f1_true_model())
    nd = 4 * 125 + 3 * T.size * 2
    dobs = vpvs_ref.vpvs_objective(oracle, x, np.zeros(nd), cfg, 0)[2]
    assert dobs.size == nd
    check_parity(ctx, oracle, cfg, models(x, 12, seed=9), dobs, which, min_ok=0.95, gmax=5e-2)


@pytest.mark.parametrize("n", [5, 12, 30, 120])
def test_every_propagator_bound_runs_the_vpvs_rows(ctx, oracle, n):
    """one n at each NMAX bound of rf_propagate_kernel (8, 16, 48, 208): each NQ = 3 instantiation"""
    rng = np.random.default_rng(n)
    vs = np.sort(rng.uniform(2.5, 4.5, n))
    thk = np.hstack((rng.uniform(0.5, 40.0 / n + 1.0, n - 1), [0.0]))
    x = x3(np.hstack((vs, thk)))
    cfg = f1_config()
    dobs = vpvs_ref.vpvs_objective(oracle, x, np.zeros(125), cfg, 1)[2]
    X = x * (1 + 0.03 * rng.uniform(-1, 1, (4, x.size)))
    X[:, 2 * n - 1] = 0.0
    check_parity(ctx, oracle, cfg, X, dobs, 1, min_ok=1.0, gmax=TOL_G)


@pytest.mark.parametrize("which", [0, 1, 2])
@pytest.mark.parametrize("method,sphere", [("freq", False), ("time", False), ("freq", True)])
def test_identity_with_the_brocher_path(oracle, which, method, sphere):
    cfg = dict(f1_config(), method=method, sphere=sphere)
    x2 = f1_true_model()
    dobs = oracle.joint_batch(x2[None, :] * 1.0, np.zeros(197), cfg)[2][0]
    rng = np.random.default_rng(3)
    X2 = x2 * (1 + 0.05 * rng.uniform(-1, 1, (32, 14)))
    X2[:, 13] = rng.uniform(0, 2, 32)
    n = 7
    vs = X2[:, :n]
    vpB = brocher(vs)[0]
    k = vpB / vs
    X3 = np.hstack((X2, k))
    sl = data_of(cfg, which)
    a, b = Context(0), Context(0)
    configure(a, n, cfg, which, vpvs=False)
    configure(b, n, cfg, which, vpvs=True)
    a.config_obs(dobs[sl])
    b.config_obs(dobs[sl])
    U2, g2, d2, f2 = a.misfit_grad_host(X2, which=which)
    U3, g3, d3, f3 = b.misfit_grad_host(X3, which=which)
    assert np.array_equal(f2, f3) and f2.sum() > 16
    m = f2
    assert np.max(np.abs(U3[m] - U2[m]) / U2[m]) <= 1e-9
    assert np.max(np.abs(d3[m] - d2[m])) <= 1e-9 * np.max(np.abs(d2[m]))
    scale = np.max(np.abs(g2[m]), axis=1, keepdims=True)
    assert np.max(np.abs(g3[m, n:2 * n] - g2[m, n:]) / scale) <= 1e-9
    dadb = 2.0947 - 0.8206 * 2 * vs + 0.2683 * 3 * vs**2 - 0.0251 * 4 * vs**3
    gvs = g3[:, :n] + g3[:, 2 * n:] * (dadb - k) / vs
    assert np.max(np.abs(gvs[m] - g2[m, :n]) / scale) <= 1e-9


def test_central_differences_in_k(ctx, oracle):
    """RF-only objective, frequency method (the SWD float32 boundary makes differences in k noisy)"""
    cfg = f1_config()
    x = x3(f1_true_model())
    dobs = vpvs_ref.vpvs_objective(oracle, x, np.zeros(125), cfg, 1)[2]
    configure(ctx, 7, cfg, 1)
    ctx.config_obs(dobs)
    xp = x * (1 + 0.03 * np.sin(np.arange(21.0)))
    xp[13] = 0.0
    _, g, _, _ = ctx.misfit_grad_host(xp[None, :], which=1)
    h = 1e-6
    E = np.eye(21)[14:] * h
    Up, _, _, _ = ctx.misfit_grad_host(xp + E, which=1)
    Um, _, _, _ = ctx.misfit_grad_host(xp - E, which=1)
    fd = (Up - Um) / (2 * h)
    assert np.max(np.abs(fd - g[0, 14:])) <= 1e-5 * np.max(np.abs(g[0, 14:]))


@pytest.mark.parametrize("which", [0, 1, 2])
def test_grouped_rows_equal_one_set_contexts_with_every_table(which):
    T = np.arange(5., 41.)
    cfg = dict(f1_config(), ray_p=[0.045, 0.06], gauss=[1.5, 2.5])
    S, n = 3, 7
    x = x3(f1_true_model())
    rng = np.random.default_rng(11)
    n1 = 4 * 125
    nd = {0: n1 + 72, 1: n1, 2: 72}[which]
    dobs = rng.normal(0, 0.05, (S, nd))
    if which != 1:
        dobs[:, nd - 72:] = 3.0 + rng.normal(0, 0.1, (S, 72))
    rays = np.array([[0.045, 0.06], [0.05, 0.07], [0.04, 0.055]])
    gauss = np.array([[1.5, 2.5], [1.0, 3.0], [2.0, 2.5]])
    use_p = np.ones((S, 72), dtype=bool)
    use_p[1, 3:10] = False
    use_p[2, 40:] = False
    use_rf = np.ones((S, n1), dtype=bool)
    use_rf[0, 125:250] = False
    use_rf[2, 10:60] = False
    X = models(x, 8, seed=13)
    sets = np.arange(X.shape[0]) % S

    def tables(c, s):
        if which != 2:
            c.config_obs_rays(rays[s])
            c.config_obs_rf_samples(use_rf[s])
            c.config_obs_gauss(gauss[s])
        if which != 1:
            c.config_obs_periods(use_p[s])

    g = Context(0)
    configure(g, n, dict(cfg, tRc=T, tRg=T.copy()), which)
    g.config_obs(dobs)
    tables(g, slice(None))
    Ug, gg, dg, fg = g.misfit_grad_host(X, which=which, sets=sets)
    assert fg.sum() > 0
    for s in range(S):
        c = Context(0)
        configure(c, n, dict(cfg, tRc=T, tRg=T.copy()), which)
        c.config_obs(dobs[s:s + 1])
        tables(c, slice(s, s + 1))
        r = sets == s
        U1, g1, d1, f1 = c.misfit_grad_host(X[r], which=which)
        assert np.array_equal(f1, fg[r]) and np.array_equal(U1, Ug[r]) and np.array_equal(g1, gg[r]), s
        assert np.array_equal(d1, dg[r], equal_nan=True), s


def _hmc_setup(oracle, which, S=1):
    cfg = f1_config()
    x = x3(f1_true_model())
    sl = data_of(cfg, which)
    dobs = np.stack([vpvs_ref.vpvs_objective(oracle, x * (1 + 0.01 * s), np.zeros(197), cfg, 0)[2][sl]
                     for s in range(S)])
    bounds = np.stack([driver_bounds_vpvs(x * (1 + 0.01 * s)) for s in range(S)])
    return cfg, dobs, bounds


@pytest.mark.parametrize("which", [0, 1, 2])
def test_base_sampler_accept_sequences(ctx, oracle, which):
    cfg, dobs, bounds = _hmc_setup(oracle, which)
    configure(ctx, 7, cfg, which)
    ctx.config_obs(dobs[0])
    ids, niter = [0, 1], 12
    out = ctx.hmc_run(0, ids, bounds[0], 0.05, Lrange=(5, 12), seed=4242, nsamples=20, ndraws=3,
                      max_iters=niter, want_samples=True, log_accepts=niter, which=which)
    assert out["samples"].shape[-1] == 21 and out["initmodel"].shape == (2, 21)
    f = vpvs_ref.oracle_vpvs_f(oracle, dobs[0], cfg, which)
    for i, cid in enumerate(ids):
        R = vpvs_ref.run_base(f, bounds[0], 0.05, (5, 12), 4242 + cid, nsamples=20, ndraws=3, max_iters=niter)
        x0 = out["initmodel"][i]
        assert np.allclose(x0, R.initmodel, rtol=0, atol=1e-14)
        assert np.all(np.diff(x0[:7]) > 0)
        seq = out["accept_seq"][i][:out["n_iter"][i]]
        assert list(seq) == R.accepts, (cid, list(seq), R.accepts)
        assert out["n_acc"][i] == R.n_acc
        ns = max(0, R.n_acc - 3)
        if ns > 0:
            assert np.allclose(out["samples"][i][:ns], R.samples[:ns], rtol=1e-6, atol=1e-9)


def test_dual_averaging_sampler_accept_sequences(ctx, oracle):
    cfg, dobs, bounds = _hmc_setup(oracle, 0)
    configure(ctx, 7, cfg, 0)
    ctx.config_obs(dobs[0])
    ids, niter = [0, 3], 8
    out = ctx.hmc_run(1, ids, bounds[0], 0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=10, ndraws=3,
                      max_iters=niter, want_samples=True, log_accepts=niter)
    f = vpvs_ref.oracle_vpvs_f(oracle, dobs[0], cfg)
    for i, cid in enumerate(ids):
        R = vpvs_ref.run_da(f, bounds[0], 0.02, 10, 0.65, 991206 + cid, nsamples=10, ndraws=3, max_iters=niter)
        assert np.allclose(out["initmodel"][i], R.initmodel, rtol=0, atol=1e-14)
        seq = out["accept_seq"][i][:out["n_iter"][i]]
        assert list(seq) == R.accepts, (cid, list(seq), R.accepts)
        assert np.isclose(out["dt"][i], R.dt, rtol=1e-6)


@pytest.mark.parametrize("sampler", [0, 1])
def test_sets_with_per_set_boxes(ctx, oracle, sampler):
    cfg, dobs, bounds = _hmc_setup(oracle, 0, S=2)
    configure(ctx, 7, cfg, 0)
    ctx.config_obs(dobs)
    ids, sets, niter = [0, 1, 0, 1], [0, 0, 1, 1], 6
    kw = dict(Lrange=(5, 10)) if sampler == 0 else dict(L0=8, target_ratio=0.65)
    dt = 0.05 if sampler == 0 else 0.02
    out = ctx.hmc_run(sampler, ids, bounds, dt, seed=77, nsamples=10, ndraws=2, max_iters=niter,
                      want_samples=True, log_accepts=niter, sets=sets, **kw)
    for i, (cid, s) in enumerate(zip(ids, sets)):
        f = vpvs_ref.oracle_vpvs_f(oracle, dobs[s], cfg)
        if sampler == 0:
            R = vpvs_ref.run_base(f, bounds[s], dt, (5, 10), 77 + cid, nsamples=10, ndraws=2, max_iters=niter)
        else:
            R = vpvs_ref.run_da(f, bounds[s], dt, 8, 0.65, 77 + cid, nsamples=10, ndraws=2, max_iters=niter)
        x0 = out["initmodel"][i]
        assert np.allclose(x0, R.initmodel, rtol=0, atol=1e-14)
        lo, hi = bounds[s][:, 0], bounds[s][:, 1]
        inside = (x0 >= lo) & (x0 <= hi)
        inside[13] = True
        assert inside.all() and np.all(np.diff(x0[:7]) > 0)
        seq = out["accept_seq"][i][:out["n_iter"][i]]
        assert list(seq) == R.accepts, (cid, s, list(seq), R.accepts)


def test_config_param_errors_and_scope(ctx):
    from rfsurfhmc_b200._lib import RfsError
    c = Context(0)
    for bad in (-1, 2, 7):
        with pytest.raises(RfsError):
            c.config_param(bad)
    cfg = f1_config()
    configure(c, 7, cfg, 1)
    x = x3(f1_true_model())
    c.config_obs(np.zeros(125))
    U3, g3, _, _ = c.misfit_grad_host(x[None, :], which=1)
    assert g3.shape == (1, 21)
    # an RF reconfiguration keeps the parameterisation; switching back restores the 2n layout
    c.config_rf(7, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"])
    assert c.misfit_grad_host(x[None, :], which=1)[1].shape == (1, 21)
    c.config_param(False)
    assert c.misfit_grad_host(x[None, :14], which=1)[1].shape == (1, 14)
