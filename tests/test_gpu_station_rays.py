"""Per-station ray parameters (rfs_config_obs_rays): every row of a grouped evaluation, and every chain
of a grouped HMC run, must give exactly what a context holding only that row's station, configured with
that station's ray parameter(s) through config_rf, gives."""
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
RAYS1 = np.array([0.045, 0.052, 0.06, 0.068, 0.075])
RAYS2 = np.array([[0.04, 0.06], [0.045, 0.065], [0.05, 0.07], [0.055, 0.062], [0.042, 0.071]])
RAYS_S = np.array([0.1, 0.105, 0.11, 0.115, 0.12])  # S-wave RF: slowness of teleseismic S

# (name, which, RF method, RF type, template ray parameter(s), per-station table)
CASES = [
    ("joint_freq", 0, "freq", "P", 0.045, RAYS1),
    ("rf_freq", 1, "freq", "P", 0.045, RAYS1),
    ("joint_time", 0, "time", "P", 0.045, RAYS1),
    ("rf_time", 1, "time", "P", 0.045, RAYS1),
    ("joint_S", 0, "freq", "S", 0.1, RAYS_S),
    ("rf_S", 1, "freq", "S", 0.1, RAYS_S),
    ("joint_two_rays", 0, "freq", "P", [0.04, 0.06], RAYS2),
]


def _configure(c, which, method="freq", rf_type="P", rays=0.045):
    cfg = f1_config()
    if which != 1:
        c.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"])
    if which != 2:
        c.config_rf(7, rays, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], rf_type, method)


def _stations(c, which, table, nsta=S, seed=3):
    """Observations of nsta stations, each forward-modelled with its own ray parameter(s): seeded
    perturbations of the F1 true model plus seeded noise (c is configured for the RF objective)."""
    c.config_obs(np.zeros((nsta, c.ndata(which))))
    c.config_obs_rays(table[:nsta])
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


def _per_station(which, method, rf_type, table, dobs, X, sets):
    """Reference: one context per station, configured with that station's ray parameter(s) through
    config_rf, evaluated on that station's rows."""
    out = [np.zeros(len(X)), np.zeros(X.shape), None, np.zeros(len(X), dtype=bool)]
    for s in range(len(dobs)):
        c = Context(0)
        try:
            p = table[s]
            _configure(c, which, method, rf_type, float(p) if np.ndim(p) == 0 else list(p))
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
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


@pytest.mark.parametrize("name,which,method,rf_type,rays,table", CASES, ids=[c[0] for c in CASES])
def test_grouped_rays_equal_per_station_contexts(name, which, method, rf_type, rays, table):
    c = Context(0)
    try:
        _configure(c, which, method, rf_type, rays)
        dobs = _stations(c, which, table)
        X, sets = _rows()
        c.config_obs(dobs, SIGMA1, SIGMA2)
        shared = c.misfit_grad_host(X, which, sets=sets)
        c.config_obs_rays(table)
        got = c.misfit_grad_host(X, which, sets=sets)
    finally:
        c.close()
    want = _per_station(which, method, rf_type, table, dobs, X, sets)
    _assert_same(got, want, name)
    ok = got[3] & shared[3]
    assert not np.array_equal(got[0][ok], shared[0][ok])  # the table is really used
    if which == 0:
        fail = ~got[3]
        assert fail.any() and fail.sum() < len(X) // 2
        # the failure convention returns the row's own station's dobs
        assert np.array_equal(got[2][fail], dobs[sets[fail]])


@pytest.mark.parametrize("which", [0, 1])
def test_chunked_batch_uses_each_chunks_own_rays(which):
    """A 1 MiB workspace budget forces about eleven 32-row chunks: each chunk's RF kernels must read
    the ray parameters of its own rows."""
    X, sets = _rows()
    plain = Context(0)
    try:
        _configure(plain, which)
        dobs = _stations(plain, which, RAYS1)
        plain.config_obs(dobs, SIGMA1, SIGMA2)
        plain.config_obs_rays(RAYS1)
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
        _configure(c, which)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_rays(RAYS1)
        n0 = c.launches
        got = c.misfit_grad_host(X, which, sets=sets)
        assert c.launches - n0 >= 8 * plain_launches  # really chunked
    finally:
        c.close()
    _assert_same(got, want, "chunked")
    _assert_same(got, _per_station(which, "freq", "P", RAYS1, dobs, X, sets), "chunked vs per station")


@pytest.mark.parametrize("which,method,rays", [(0, "freq", 0.045), (1, "time", 0.045), (1, "freq", [0.04, 0.06])])
def test_table_of_the_shared_value_gives_the_same_bits(which, method, rays):
    c = Context(0)
    try:
        _configure(c, which, method, "P", rays)
        dobs = _stations(c, which, RAYS1 if np.ndim(rays) == 0 else RAYS2)
        X, sets = _rows(B=160, seed=11)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        want = c.misfit_grad_host(X, which, sets=sets)
        c.config_obs_rays(np.tile(np.atleast_1d(rays), (S, 1)))
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


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "freq"), (1, "time")])
def test_out_of_range_set_fails_only_its_row(which, method):
    c = Context(0)
    try:
        _configure(c, which, method)
        dobs = _stations(c, which, RAYS1)
        X, sets = _rows(B=96, seed=4)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_rays(RAYS1)
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


def test_config_obs_rays_errors():
    c = Context(0)
    try:
        _configure(c, 2)  # SWD only: no RF configuration
        c.config_obs(np.zeros((S, c.ndata(2))))
        with pytest.raises(RfsError) as e:
            c.config_obs_rays(RAYS1)
        assert e.value.code == RFS_E_CONFIG
    finally:
        c.close()
    c = Context(0)
    try:
        _configure(c, 1)
        with pytest.raises(RfsError) as e:  # no observation sets yet
            c.config_obs_rays(RAYS1)
        assert e.value.code == RFS_E_CONFIG
        c.config_obs(np.zeros((S, c.ndata(1))))
        with pytest.raises(RfsError) as e:  # S differs from the sets held
            c.config_obs_rays(RAYS1[:S - 1])
        assert e.value.code == RFS_E_CONFIG
        with pytest.raises(RfsError) as e:  # two rays for a one-ray objective
            c.config_obs_rays(RAYS2)
        assert e.value.code == RFS_E_ARG
        for v in (0.0, -0.05, np.nan, np.inf):
            t = RAYS1.copy()
            t[2] = v
            with pytest.raises(RfsError) as e:
                c.config_obs_rays(t)
            assert e.value.code == RFS_E_ARG, v
        c.config_obs_rays(RAYS1)
    finally:
        c.close()


def test_every_config_call_drops_the_table():
    """After rfs_config_obs_sets, rfs_config_obs, rfs_config_rf and rfs_config_rf_rays, the context
    computes with the shared ray parameter again."""
    cfg = f1_config()
    X, sets = _rows(B=64, seed=9)
    c = Context(0)
    try:
        _configure(c, 0)
        dobs = _stations(c, 0, RAYS1)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        shared = c.misfit_grad_host(X, 0, sets=sets)
        c.config_obs_rays(RAYS1)
        table = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(table[0], shared[0])
        # rfs_config_obs_sets
        c.config_obs(dobs, SIGMA1, SIGMA2)
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), shared, "config_obs_sets")
        # rfs_config_rf_rays
        c.config_obs_rays(RAYS1)
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "table again")
        _configure(c, 1)
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), shared, "config_rf_rays")
        # rfs_config_rf (the scalar call)
        c.config_obs_rays(RAYS1)
        rc = c.L.rfs_config_rf(c.h, 7, ctypes.c_double(cfg["ray_p"]), cfg["nt"], cfg["dt"], cfg["gauss"],
                               cfg["time_shift"], cfg["water"], 1, 1)
        assert rc == 0
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), shared, "config_rf")
        # rfs_config_obs (the one-set call)
        one = sets == 3
        c.config_obs(dobs[3], SIGMA1[3], SIGMA2[3])
        want = c.misfit_grad_host(X[one], 0)
        c.config_obs_rays(RAYS1[3:4])
        assert not np.array_equal(c.misfit_grad_host(X[one], 0)[0], want[0])
        d3 = np.ascontiguousarray(dobs[3])
        rc = c.L.rfs_config_obs(c.h, SIGMA1[3], SIGMA2[3], d3.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                d3.size)
        assert rc == 0
        _assert_same(c.misfit_grad_host(X[one], 0), want, "config_obs")
    finally:
        c.close()


def _boxes(nsta):
    b = np.repeat(driver_bounds(f1_true_model())[None], nsta, axis=0)
    for s in range(nsta):
        b[s, :7, 0] *= 1.0 + 0.04 * s
        b[s, :7, 1] *= 1.0 - 0.03 * s
    return b


@pytest.mark.parametrize("sampler", [0, 1])
def test_hmc_over_stations_with_rays_equals_single_station_runs(sampler):
    nsta, K = 3, 6
    kw = (dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=6, ndraws=1, max_iters=14) if sampler == 0 else
          dict(dt=0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=3, ndraws=3, max_iters=14))
    kw.update(want_samples=True, log_accepts=kw["max_iters"])
    boxes = _boxes(nsta)
    c = Context(0)
    try:
        _configure(c, 0)
        dobs = _stations(c, 0, RAYS1, nsta, seed=5)
    finally:
        c.close()
    want = {}
    for s in range(nsta):
        c = Context(0)
        try:
            _configure(c, 0, rays=float(RAYS1[s]))
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
            want[s] = c.hmc_run(sampler, np.arange(K), boxes[s], **kw)
        finally:
            c.close()
    c = Context(0)
    try:
        _configure(c, 0)
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        c.config_obs_rays(RAYS1[:nsta])
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


def _f1_models(rays):
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    cfg = f1_config()
    rf = ReceiverFunc(rays, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                      cfg["rf_type"], cfg["method"])
    swd = SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"])
    return Joint_RF_SWD(1.0, 1.0, rf, swd)


def test_station_array_with_rays_matches_its_station_models(tmp_path):
    from rfsurfhmc_b200.model.stations import StationArray
    from rfsurfhmc_b200.pyhmc.hmc import HamitonianMC
    c = Context(0)
    try:
        _configure(c, 0)
        dobs = _stations(c, 0, RAYS1, 2, seed=6)
    finally:
        c.close()
    sa = StationArray(_f1_models(0.045), dobs, sigma1=[1.0, 0.5], names=["AA01", "BB02"], ray_p=RAYS1[:2])
    X, _ = _rows(B=16, seed=2, nsta=2)
    got = sa.misfit_and_grad_batch(X, np.arange(16) % 2)
    for s in range(2):
        m = sa.station_model(s)
        assert m.rfmodel.ray_p == RAYS1[s]
        for a, b in zip(got, m.misfit_and_grad_batch(X[s::2])):
            assert np.array_equal(a[s::2], b, equal_nan=True)
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


def test_driver_runs_a_stations_file_with_rays(tmp_path):
    from rfsurfhmc_b200 import driver
    with open(os.path.join(ROOT, "tests", "golden", "f1_param.yaml")) as fh:
        param = yaml.safe_load(fh)
    c = Context(0)
    try:
        _configure(c, 0, rays=param["rf"]["ray_p"])
        dobs = _stations(c, 0, RAYS1[2:], 2, seed=7)
    finally:
        c.close()

    def run(tag, **keys):
        param["hmc"].update(OUTPUT_DIR=str(tmp_path / tag), nsamples=3, ndraws=1)
        path = tmp_path / f"{tag}.npz"
        np.savez(path, **keys)
        return driver.run(param, "base", 2, save_chains=False, max_iters=8, stations=str(path))[0]

    both = run("both", dobs=dobs, names=np.array(["N1", "N2"]), ray_p=RAYS1[2:4])
    alone = run("alone", dobs=dobs[1:], names=np.array(["N2"]), ray_p=RAYS1[3:4])
    shared = run("shared", dobs=dobs, names=np.array(["N1", "N2"]))
    assert np.array_equal(np.load(tmp_path / "both" / "N2" / "misfit.npy"), both[2:], equal_nan=True)
    assert np.array_equal(both[2:], alone, equal_nan=True)
    assert not np.array_equal(both[2:], shared[2:], equal_nan=True)


def test_joint_evaluator_with_obs_ray_p():
    from rfsurfhmc_b200.batched import JointEvaluator
    cfg = f1_config()
    cfg.update(sigma1=SIGMA1, sigma2=SIGMA2)
    c = Context(0)
    try:
        _configure(c, 0)
        dobs = _stations(c, 0, RAYS1)
        X, sets = _rows(B=128, seed=12)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        c.config_obs_rays(RAYS1)
        want = c.misfit_grad_host(X, 0, sets=sets)
    finally:
        c.close()
    ev = JointEvaluator(cfg, dobs, 7, obs_ray_p=RAYS1)
    dev = torch.device("cuda", 0)
    U, G, D, F = ev(torch.from_numpy(X).to(dev), torch.from_numpy(sets).to(dev))
    torch.cuda.synchronize(dev)
    got = [U.cpu().numpy(), G.cpu().numpy(), D.cpu().numpy(), F.cpu().numpy().astype(bool)]
    ev.ctx.close()
    _assert_same(got, want, "JointEvaluator")
