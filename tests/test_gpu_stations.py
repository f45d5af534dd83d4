"""Many observation sets (stations) in one context: every row of a grouped evaluation, and every chain
of a grouped HMC run, must give exactly what a context holding only that row's station gives."""
import os
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

# (name, which, RF method, SWD modes, ray parameters)
CASES = [
    ("joint_freq", 0, "freq", 0, None),
    ("rf_freq", 1, "freq", 0, None),
    ("swd", 2, "freq", 0, None),
    ("joint_time", 0, "time", 0, None),
    ("rf_time", 1, "time", 0, None),
    ("joint_modes_rays", 0, "freq", [0, 1], [0.04, 0.06]),
]


def _configure(c, which, method, modes, rays):
    cfg = f1_config()
    if which != 1:
        c.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"], mode=modes)
    if which != 2:
        c.config_rf(7, cfg["ray_p"] if rays is None else rays, cfg["nt"], cfg["dt"], cfg["gauss"],
                    cfg["time_shift"], cfg["water"], cfg["rf_type"], method)


def _stations(c, which, nsta=S, seed=3):
    """Observations of nsta stations: the forward model of seeded perturbations of the F1 true model
    plus seeded noise (c is configured, with any observations of the right length)."""
    c.config_obs(np.zeros(c.ndata(which)))
    Xs = perturbed_models(f1_true_model(), nsta, seed=seed, rel=0.05)
    _, _, d, _ = c.misfit_grad_host(Xs, which)
    # a higher mode that does not exist at a period has a NaN synthetic; a measured data vector has a
    # number there, so that the misfits compared below are finite
    d = np.where(np.isfinite(d), d, 0.0)
    return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)


def _rows(B=333, seed=8):
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
    sets = rng.integers(0, S, B).astype(np.int32)
    sets[:S] = np.arange(S)
    return X, sets


def _per_station(which, method, modes, rays, dobs, X, sets):
    """Reference result: one context holding one station at a time, evaluated on that station's rows."""
    c = Context(0)
    try:
        _configure(c, which, method, modes, rays)
        nd = c.ndata(which)
        out = [np.zeros(len(X)), np.zeros(X.shape), np.zeros((len(X), nd)), np.zeros(len(X), dtype=bool)]
        for s in range(S):
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
            r = sets == s
            for o, v in zip(out, c.misfit_grad_host(X[r], which)):
                o[r] = v
        return out
    finally:
        c.close()


def _grouped(c, which, dobs, X, sets):
    c.config_obs(dobs, SIGMA1, SIGMA2)
    return c.misfit_grad_host(X, which, sets=sets)


def _assert_same(got, want, tag):
    for name, a, b in zip(("U", "grad", "dsyn", "flag"), got, want):
        assert np.array_equal(a, b, equal_nan=True), (tag, name)


@pytest.mark.parametrize("name,which,method,modes,rays", CASES, ids=[c[0] for c in CASES])
def test_grouped_evaluation_equals_per_station(name, which, method, modes, rays):
    c = Context(0)
    try:
        _configure(c, which, method, modes, rays)
        dobs = _stations(c, which)
        X, sets = _rows()
        got = _grouped(c, which, dobs, X, sets)
    finally:
        c.close()
    want = _per_station(which, method, modes, rays, dobs, X, sets)
    _assert_same(got, want, name)
    if which != 1:
        fail = ~got[3]
        assert fail.any() and fail.sum() < len(X) // 2
        # the reference's failure convention returns the row's own station's dobs (zeros for SWD only)
        exp = dobs[sets[fail]] if which == 0 else np.zeros((int(fail.sum()), dobs.shape[1]))
        assert np.array_equal(got[2][fail], exp)


@pytest.mark.parametrize("which", [0, 1])
def test_chunked_batch_reads_each_chunks_own_sets(which):
    """A 1 MiB workspace budget forces the 32-row floor of the chunk size: the 333 rows run in about
    eleven chunks, each of which must read its own slice of the set array."""
    X, sets = _rows()
    plain = Context(0)
    try:
        _configure(plain, which, "freq", 0, None)
        dobs = _stations(plain, which)
        n0 = plain.launches
        want = _grouped(plain, which, dobs, X, sets)
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
        _configure(c, which, "freq", 0, None)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        n0 = c.launches
        got = c.misfit_grad_host(X, which, sets=sets)
        assert c.launches - n0 >= 8 * plain_launches  # really chunked
    finally:
        c.close()
    _assert_same(got, want, "chunked")
    _assert_same(got, _per_station(which, "freq", 0, None, dobs, X, sets), "chunked vs per station")


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "freq"), (2, "freq"), (1, "time")])
def test_out_of_range_set_indices(which, method):
    c = Context(0)
    try:
        _configure(c, which, method, 0, None)
        dobs = _stations(c, which)
        X, sets = _rows(B=96, seed=4)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        for bad in (-1, S):
            s = sets.copy()
            s[7] = bad
            with pytest.raises(RfsError) as e:
                c.misfit_grad_host(X, which, sets=s)
            assert e.value.code == RFS_E_ARG
        want = c.misfit_grad_host(X, which, sets=sets)
        # device API: no check without a synchronise; the bad rows read nothing and are marked failed
        s = sets.copy()
        bad = np.array([3, 40, 95])
        s[bad] = [-1, S, 1 << 30]
        dev = torch.device("cuda", 0)
        xd = torch.from_numpy(X).to(dev)
        sd = torch.from_numpy(s).to(dev)
        nd = c.ndata(which)
        U = torch.full((len(X),), 7.0, dtype=torch.float64, device=dev)
        G = torch.full((len(X), X.shape[1]), 7.0, dtype=torch.float64, device=dev)
        D = torch.zeros((len(X), nd), dtype=torch.float64, device=dev)
        F = torch.full((len(X),), 9, dtype=torch.uint8, device=dev)
        st = torch.cuda.current_stream(dev)
        c.misfit_grad_dev(len(X), xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                          st.cuda_stream, sets_ptr=sd.data_ptr())
        st.synchronize()
        got = [U.cpu().numpy(), G.cpu().numpy(), D.cpu().numpy(), F.cpu().numpy().astype(bool)]
        assert (got[0][bad] == 0).all() and (got[1][bad] == 0).all() and np.isnan(got[2][bad]).all()
        assert not got[3][bad].any() and set(F.cpu().numpy().tolist()) <= {0, 1}
        ok = np.setdiff1d(np.arange(len(X)), bad)
        for name, a, b in zip(("U", "grad", "dsyn", "flag"), got, want):
            assert np.array_equal(a[ok], b[ok], equal_nan=True), name
        # calls without a set array on a context holding several sets
        with pytest.raises(RfsError) as e:
            c.misfit_grad_host(X, which)
        assert e.value.code == RFS_E_CONFIG and "rfs_misfit_grad_sets" in str(e.value)
        bounds = driver_bounds(f1_true_model())
        with pytest.raises(RfsError) as e:
            c.hmc_run(0, [0, 1], bounds, 0.1, nsamples=2, ndraws=1, max_iters=2, which=which)
        assert e.value.code == RFS_E_CONFIG and "rfs_hmc_run_sets" in str(e.value)
        with pytest.raises(RfsError) as e:
            c.hmc_run(0, [0, 1], bounds, 0.1, nsamples=2, ndraws=1, max_iters=2, which=which, sets=[0, S])
        assert e.value.code == RFS_E_ARG
    finally:
        c.close()


def _boxes(nsta):
    """A different search box per station."""
    b = np.repeat(driver_bounds(f1_true_model())[None], nsta, axis=0)
    for s in range(nsta):
        b[s, :7, 0] *= 1.0 + 0.04 * s
        b[s, :7, 1] *= 1.0 - 0.03 * s
    return b


@pytest.mark.parametrize("sampler", [0, 1])
def test_hmc_over_stations_equals_per_station_runs(sampler):
    nsta, K = 3, 6
    kw = (dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=6, ndraws=1, max_iters=14) if sampler == 0 else
          dict(dt=0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=3, ndraws=3, max_iters=14))
    kw.update(want_samples=True, log_accepts=kw["max_iters"])
    boxes = _boxes(nsta)
    c = Context(0)
    try:
        _configure(c, 0, "freq", 0, None)
        dobs = _stations(c, 0, nsta, seed=5)
        want = {}
        for s in range(nsta):
            c.config_obs(dobs[s], SIGMA1[s], SIGMA2[s])
            want[s] = c.hmc_run(sampler, np.arange(K), boxes[s], **kw)
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
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
            for s in range(nsta):  # every initial model lies in its own station's box
                ini = got["initmodel"][sets == s]
                assert (ini >= boxes[s][:, 0]).all() and (ini <= boxes[s][:, 1]).all()
    finally:
        c.set_hmc_options(resident=0)
        c.close()


def _f1_models():
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    cfg = f1_config()
    rf = ReceiverFunc(cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                      cfg["rf_type"], cfg["method"])
    swd = SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"])
    return Joint_RF_SWD(1.0, 1.0, rf, swd)


def test_station_array_sampler_writes_per_station_files(tmp_path):
    from rfsurfhmc_b200.model.stations import StationArray
    from rfsurfhmc_b200.pyhmc.hmc import HamitonianMC
    model = _f1_models()
    c = Context(0)
    try:
        _configure(c, 0, "freq", 0, None)
        dobs = _stations(c, 0, 2, seed=6)
    finally:
        c.close()
    sa = StationArray(model, dobs, sigma1=[1.0, 0.5], names=["AA01", "BB02"])
    X, _ = _rows(B=16, seed=2)
    U, g, d, f = sa.misfit_and_grad_batch(X, np.arange(16) % 2)
    one = sa.station_model(1).misfit_and_grad_batch(X[1::2])
    for a, b in zip((U[1::2], g[1::2], d[1::2], f[1::2]), one):
        assert np.array_equal(a, b)
    hmc = HamitonianMC(sa, driver_bounds(f1_true_model()), 0.1, (5, 20), 3, 991206, 4, 1, name="ch",
                       outdir=str(tmp_path))
    hmc.max_iters = 12
    out = hmc.sample_chains([0, 1, 0], stations=[0, 0, 1], save=True)
    assert out["station"].tolist() == [0, 0, 1]
    for s, cid in ((0, 0), (0, 1), (1, 0)):
        z = np.load(tmp_path / sa.names[s] / f"ch.{cid}.npz")
        assert np.array_equal(z["obs"], dobs[s])


def test_driver_runs_a_stations_file(tmp_path):
    from rfsurfhmc_b200 import driver
    with open(os.path.join(ROOT, "tests", "golden", "f1_param.yaml")) as fh:
        param = yaml.safe_load(fh)
    param["hmc"].update(OUTPUT_DIR=str(tmp_path / "out"), nsamples=3, ndraws=1)
    c = Context(0)
    try:
        _configure(c, 0, "freq", 0, None)
        dobs = _stations(c, 0, 2, seed=7)
    finally:
        c.close()
    path = tmp_path / "stations.npz"
    np.savez(path, dobs=dobs, names=np.array(["N1", "N2"]), bounds=_boxes(2))
    misfit, n_iter, out = driver.run(param, "base", 2, save_chains=True, max_iters=8, stations=str(path))
    assert misfit.shape == (4, 3)
    for s, name in enumerate(("N1", "N2")):
        m = np.load(tmp_path / "out" / name / "misfit.npy")
        assert m.shape == (2, 3)
        assert np.array_equal(m, misfit[2 * s:2 * s + 2], equal_nan=True)
        assert (tmp_path / "out" / name / "chain_joint.1.npz").exists()
