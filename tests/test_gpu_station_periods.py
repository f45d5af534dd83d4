"""Per-station SWD period lists (rfs_config_obs_periods): every row of a grouped evaluation, and every
chain of a grouped HMC run, must give exactly what a context holding only that row's station, configured
through config_swd on that station's subset period lists, gives.  dsyn keeps the grid layout: the
subset context's values at the observed periods, NaN at the others."""
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
T = np.arange(5., 41.)
F1 = dict(lists=(T, T.copy(), [], []), modes=0, sphere=False, n=7)
# Love and Rayleigh on four different grids, modes 0-2, earth flattening
LR = dict(lists=(T[::2], T[1::3], np.arange(6., 30., 2.), np.arange(8., 36., 3.)), modes=[0, 1, 2], sphere=True, n=7)
N40 = dict(lists=(np.geomspace(2, 100, 24), np.geomspace(3, 80, 18), [], []), modes=[0, 1, 2], sphere=False, n=40)


def _x40_true():
    i = np.arange(40)
    vs = 2.0 + 2.7 * (i / 39.0) ** 0.7
    thk = np.hstack((0.5 + 0.1 * i[:-1], [0.0]))
    return np.hstack((vs, thk))


def _x0(case):
    return f1_true_model() if case["n"] == 7 else _x40_true()


def _window(rng, n):
    """Contiguous window of 60-100 % of n periods."""
    k = int(rng.integers(int(np.ceil(0.6 * n)), n + 1))
    a = int(rng.integers(0, n - k + 1))
    m = np.zeros(n, dtype=bool)
    m[a:a + k] = True
    return m


def _masks(case, nsta=S, seed=1, same_rc_rg=False, no_rg=None):
    """Seeded windows of every list per station; same_rc_rg: Rg observed where Rc is (the plan keeps its
    shared sequence); no_rg: a station without group-velocity data."""
    rng = np.random.default_rng(seed)
    rows = []
    for s in range(nsta):
        parts = []
        for w, t in enumerate(case["lists"]):
            if len(t) == 0:
                continue
            if w == 1 and same_rc_rg:
                parts.append(parts[0].copy())
            elif w == 1 and s == no_rg:
                parts.append(np.zeros(len(t), dtype=bool))
            else:
                parts.append(_window(rng, len(t)))
        rows.append(np.concatenate(parts))
    return np.array(rows)


def _subset(case, u):
    out, o = [], 0
    for t in case["lists"]:
        t = np.asarray(t, dtype=np.float64)
        out.append(t[u[o:o + t.size]])
        o += t.size
    return out


def _nmodes(case):
    return np.size(case["modes"])


def _configure(c, case, which, lists=None, rays=0.045):
    cfg = f1_config()
    if which != 1:
        c.config_swd(case["n"], *(case["lists"] if lists is None else lists), mode=case["modes"],
                     sphere=case["sphere"])
    if which != 2:
        c.config_rf(case["n"], rays, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                    cfg["rf_type"], cfg["method"])


def _stations(case, which, nsta=S, seed=3):
    """Grid-layout observations of nsta stations: seeded perturbations of the true model plus noise."""
    c = Context(0)
    try:
        _configure(c, case, which)
        c.config_obs(np.zeros((nsta, c.ndata(which))))
        Xs = perturbed_models(_x0(case), nsta, seed=seed, rel=0.05)
        _, _, d, _ = c.misfit_grad_host(Xs, which, sets=np.arange(nsta))
    finally:
        c.close()
    d = np.where(np.isfinite(d), d, 0.0)
    return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)


def _rows(case, B=333, seed=8, nsta=S):
    """Models near the truth, strongly perturbed ones and ones with a slow half-space (many of those
    fail the main root search and go through the per-period retries), each row on a random station."""
    x0 = _x0(case)
    n = x0.size // 2
    X = perturbed_models(x0, B, seed=seed, rel=0.1)
    rng = np.random.default_rng(seed)
    kind = rng.random(B)
    wild = kind < 0.2
    X[wild] = rng.uniform(0.5, 1.5, (int(wild.sum()), x0.size)) * x0 + 0.01
    slow = kind > 0.85
    X[slow, n - 1] = rng.uniform(1.0, 2.5, int(slow.sum()))
    sets = rng.integers(0, nsta, B).astype(np.int32)
    sets[:nsta] = np.arange(nsta)
    return X, sets


def _rf_len(which):
    return f1_config()["nt"] if which == 0 else 0


def _compact(case, which, d, u):
    nt = _rf_len(which)
    return np.concatenate([d[:nt], d[nt:][np.tile(u, _nmodes(case))]])


def _per_station(case, which, use, dobs, X, sets, rays=None):
    """Reference: one context per station, configured on that station's subset lists (and ray
    parameter), evaluated on that station's rows; dsyn scattered into the grid layout."""
    nt = _rf_len(which)
    nd = dobs.shape[1]
    out = [np.zeros(len(X)), np.zeros(X.shape), np.full((len(X), nd), np.nan), np.zeros(len(X), dtype=bool)]
    for s in range(len(dobs)):
        r = sets == s
        if not r.any():
            continue
        c = Context(0)
        try:
            _configure(c, case, which, _subset(case, use[s]), 0.045 if rays is None else float(rays[s]))
            c.config_obs(_compact(case, which, dobs[s], use[s]), SIGMA1[s], SIGMA2[s])
            U, g, d, f = c.misfit_grad_host(X[r], which)
        finally:
            c.close()
        full = np.full((int(r.sum()), nd), np.nan)
        full[:, :nt] = d[:, :nt]
        full[:, nt + np.flatnonzero(np.tile(use[s], _nmodes(case)))] = d[:, nt:]
        full[~f] = dobs[s] if which == 0 else 0.0  # the failure convention on the grid layout
        out[0][r], out[1][r], out[2][r], out[3][r] = U, g, full, f
    return out


def _grouped(case, which, use, dobs, X, sets, rays=None, team=None, sched=None, ctx=None):
    c = Context(0) if ctx is None else ctx
    try:
        _configure(c, case, which)
        if team is not None:
            c.set_roots_team(team)
        if sched is not None:
            c.set_roots_sched(sched)
        c.config_obs(dobs, SIGMA1[:len(dobs)], SIGMA2[:len(dobs)])
        if rays is not None:
            c.config_obs_rays(rays[:len(dobs)])
        if use is not None:
            c.config_obs_periods(use)
        got = c.misfit_grad_host(X, which, sets=sets)
        return got, c.last_roots_team(), c.last_roots_sched()
    finally:
        if ctx is None:
            c.close()


def _assert_same(got, want, tag, rows=slice(None)):
    for name, a, b in zip(("U", "grad", "dsyn", "flag"), got, want):
        assert np.array_equal(a[rows], b[rows], equal_nan=True), (tag, name)


# (name, case, which, mask options, rows, root-search mapping: team (None = automatic), expected T / sorted)
CASES = [
    ("f1_joint", F1, 0, dict(no_rg=2), 333, None, "team", 0),
    ("f1_swd", F1, 2, dict(no_rg=2), 333, None, "team", 0),
    ("f1_joint_shared_seq", F1, 0, dict(same_rc_rg=True), 333, None, "team", 0),
    ("f1_joint_team64", F1, 0, dict(), 64, None, "team", 0),
    ("f1_joint_thread", F1, 0, dict(no_rg=1), 1024, 0, "thread", 0),
    ("f1_joint_sorted", F1, 0, dict(no_rg=4), 8192, None, "thread", 1),
    ("love_rayleigh_modes_sphere", LR, 0, dict(), 333, None, "team", 0),
    ("n40_swd_modes_thread", N40, 2, dict(no_rg=3), 200, 0, "thread", 0),
    ("n40_swd_modes_team", N40, 2, dict(), 96, None, "team", 0),
]


@pytest.mark.parametrize("name,case,which,mopt,B,team,mapping,sorted_", CASES, ids=[c[0] for c in CASES])
def test_grouped_periods_equal_per_station_contexts(name, case, which, mopt, B, team, mapping, sorted_):
    use = _masks(case, **mopt)
    dobs = _stations(case, which)
    X, sets = _rows(case, B)
    got, (Tm, _), srt = _grouped(case, which, use, dobs, X, sets, team=team)
    assert (Tm == 0) == (mapping == "thread") and srt == sorted_, (Tm, srt)
    want = _per_station(case, which, use, dobs, X, sets)
    _assert_same(got, want, name)
    # some rows fail the main pass (a failed row had ierr != 0 and went through the per-period retries),
    # most succeed; ok rows are NaN exactly at the periods their station does not observe
    fail = ~got[3]
    assert fail.any() and fail.sum() < len(X) // 2
    nt = _rf_len(which)
    miss = ~np.tile(use, _nmodes(case))[sets]
    assert np.isnan(got[2][:, nt:][~fail][miss[~fail]]).all()
    if which == 0:
        assert np.array_equal(got[2][fail], dobs[sets[fail]])


def test_all_ones_mask_gives_the_bits_of_no_table():
    for case, which in ((F1, 0), (F1, 2), (LR, 0)):
        dobs = _stations(case, which)
        X, sets = _rows(case, 160, seed=11)
        nper = sum(len(t) for t in case["lists"])
        want, _, _ = _grouped(case, which, None, dobs, X, sets)
        got, _, _ = _grouped(case, which, np.ones((S, nper), dtype=bool), dobs, X, sets)
        _assert_same(got, want, f"all ones {which}")


def test_rf_only_evaluation_ignores_the_table():
    nt = _rf_len(0)
    dobs = _stations(F1, 0)[:, :nt]
    X, sets = _rows(F1, 96, seed=5)
    c = Context(0)
    try:
        _configure(c, F1, 0)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        want = c.misfit_grad_host(X, 1, sets=sets)
        c.config_obs_periods(_masks(F1, no_rg=0))
        _assert_same(c.misfit_grad_host(X, 1, sets=sets), want, "rf only")
    finally:
        c.close()


@pytest.mark.parametrize("which", [0, 2])
def test_chunked_batch_uses_each_chunks_own_periods(which):
    """A 1 MiB workspace budget forces many 32-row chunks: each chunk's root searches, eigen solves and
    assembly must read the period lists of its own rows."""
    use = _masks(F1, no_rg=2)
    dobs = _stations(F1, which)
    X, sets = _rows(F1)
    plain = Context(0)
    try:
        n0 = plain.launches
        want, _, _ = _grouped(F1, which, use, dobs, X, sets, ctx=plain)
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
        n0 = c.launches
        got, _, _ = _grouped(F1, which, use, dobs, X, sets, ctx=c)
        assert c.launches - n0 >= 8 * plain_launches  # really chunked
    finally:
        c.close()
    _assert_same(got, want, "chunked")
    _assert_same(got, _per_station(F1, which, use, dobs, X, sets), "chunked vs per station")


def test_periods_with_a_ray_table():
    use = _masks(F1, no_rg=3, seed=4)
    c = Context(0)
    try:
        _configure(c, F1, 0)
        c.config_obs(np.zeros((S, c.ndata(0))))
        c.config_obs_rays(RAYS1)
        _, _, d, _ = c.misfit_grad_host(perturbed_models(f1_true_model(), S, seed=2, rel=0.05), 0, sets=np.arange(S))
    finally:
        c.close()
    dobs = np.where(np.isfinite(d), d, 0.0)
    X, sets = _rows(F1, 200, seed=6)
    got, _, _ = _grouped(F1, 0, use, dobs, X, sets, rays=RAYS1)
    _assert_same(got, _per_station(F1, 0, use, dobs, X, sets, rays=RAYS1), "rays + periods")


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


@pytest.mark.parametrize("which", [0, 2])
def test_out_of_range_set_fails_only_its_row(which):
    use = _masks(F1, no_rg=1)
    dobs = _stations(F1, which)
    X, sets = _rows(F1, 96, seed=4)
    c = Context(0)
    try:
        want, _, _ = _grouped(F1, which, use, dobs, X, sets, ctx=c)
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


def _raw(c, S_, use):
    u = np.ascontiguousarray(use, dtype=np.uint8)
    return c.L.rfs_config_obs_periods(c.h, S_, u.shape[1], u.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)))


def test_config_obs_periods_errors():
    use = _masks(F1)
    c = Context(0)
    try:
        _configure(c, F1, 1)  # RF only: no SWD configuration
        c.config_obs(np.zeros((S, c.ndata(1))))
        with pytest.raises(RfsError) as e:
            c.config_obs_periods(use)
        assert e.value.code == RFS_E_CONFIG
    finally:
        c.close()
    dobs = _stations(F1, 0)
    X, sets = _rows(F1, 64, seed=9)
    c = Context(0)
    try:
        _configure(c, F1, 0)
        with pytest.raises(RfsError) as e:  # no observation sets yet
            c.config_obs_periods(use)
        assert e.value.code == RFS_E_CONFIG
        c.config_obs(dobs, SIGMA1, SIGMA2)
        grid = c.misfit_grad_host(X, 0, sets=sets)
        with pytest.raises(RfsError) as e:  # S differs from the sets held
            c.config_obs_periods(use[:S - 1])
        assert e.value.code == RFS_E_CONFIG
        with pytest.raises(RfsError) as e:  # wrong nper
            c.config_obs_periods(use[:, 1:])
        assert e.value.code == RFS_E_ARG
        bad = use.astype(np.uint8)
        bad[2, 4] = 2
        assert _raw(c, S, bad) == RFS_E_ARG
        bad = use.copy()
        bad[3] = False
        with pytest.raises(RfsError) as e:  # a station observing nothing
            c.config_obs_periods(bad)
        assert e.value.code == RFS_E_ARG
        # a failed call leaves no table, also after a valid one (and restores the shared sequence)
        c.config_obs_periods(_masks(F1, no_rg=1))
        assert _raw(c, S, bad) == RFS_E_ARG
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), grid, "failed call")
    finally:
        c.close()


def test_every_config_call_drops_the_table():
    """After rfs_config_obs_sets, rfs_config_obs, rfs_config_swd and rfs_config_swd_modes the context
    evaluates on the grid lists again; rfs_config_rf keeps the table and the joint weight follows n1."""
    cfg = f1_config()
    use = _masks(F1, no_rg=2)
    dobs = _stations(F1, 0)
    X, sets = _rows(F1, 64, seed=9)
    c = Context(0)
    try:
        _configure(c, F1, 0)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        grid = c.misfit_grad_host(X, 0, sets=sets)
        c.config_obs_periods(use)
        table = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(table[0], grid[0])
        c.config_obs(dobs, SIGMA1, SIGMA2)  # rfs_config_obs_sets
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), grid, "config_obs_sets")
        c.config_obs_periods(use)
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "table again")
        _configure(c, F1, 2)  # rfs_config_swd_modes
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), grid, "config_swd_modes")
        c.config_obs_periods(use)
        t = np.ascontiguousarray(T)
        tp = t.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        assert c.L.rfs_config_swd(c.h, 7, t.size, tp, t.size, tp, 0, None, 0, None, 0, 0, 1) == 0
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), grid, "config_swd")
        # rfs_config_rf keeps the table; a second ray doubles n1 and the weights follow
        c.config_obs_periods(use)
        _configure(c, F1, 1)
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), table, "config_rf keeps")
        c.config_rf(7, [0.045, 0.05], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"])
        nt = cfg["nt"]
        d2 = np.hstack((dobs[:, :nt], dobs[:, :nt], dobs[:, nt:]))
        c.config_obs(d2, SIGMA1, SIGMA2)
        c.config_obs_periods(use)
        two = c.misfit_grad_host(X, 0, sets=sets)
        r = sets == 1
        one = Context(0)
        try:
            one.config_swd(7, *_subset(F1, use[1])[:2])
            one.config_rf(7, [0.045, 0.05], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"])
            one.config_obs(np.concatenate((d2[1, :2 * nt], dobs[1, nt:][use[1]])), SIGMA1[1], SIGMA2[1])
            w = one.misfit_grad_host(X[r], 0)
        finally:
            one.close()
        assert np.array_equal(two[0][r], w[0]) and np.array_equal(two[1][r], w[1])
        # rfs_config_obs (the one-set call)
        c.config_obs(d2[1], SIGMA1[1], SIGMA2[1])
        plain = c.misfit_grad_host(X[r], 0)
        c.config_obs_periods(use[1:2])
        assert np.array_equal(c.misfit_grad_host(X[r], 0)[0], w[0])
        d1 = np.ascontiguousarray(d2[1])
        assert c.L.rfs_config_obs(c.h, SIGMA1[1], SIGMA2[1], d1.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                  d1.size) == 0
        _assert_same(c.misfit_grad_host(X[r], 0), plain, "config_obs")
    finally:
        c.close()


def _boxes(nsta):
    b = np.repeat(driver_bounds(f1_true_model())[None], nsta, axis=0)
    for s in range(nsta):
        b[s, :7, 0] *= 1.0 + 0.04 * s
        b[s, :7, 1] *= 1.0 - 0.03 * s
    return b


@pytest.mark.parametrize("sampler", [0, 1])
def test_hmc_over_stations_with_periods_equals_single_station_runs(sampler):
    nsta, K = 3, 6
    kw = (dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=6, ndraws=1, max_iters=14) if sampler == 0 else
          dict(dt=0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=3, ndraws=3, max_iters=14))
    kw.update(want_samples=True, want_syn=True, log_accepts=kw["max_iters"])
    boxes = _boxes(nsta)
    use = _masks(F1, nsta, seed=7, no_rg=1)
    dobs = _stations(F1, 0, nsta, seed=5)
    nt = _rf_len(0)
    want = {}
    for s in range(nsta):
        c = Context(0)
        try:
            _configure(c, F1, 0, _subset(F1, use[s]))
            c.config_obs(_compact(F1, 0, dobs[s], use[s]), SIGMA1[s], SIGMA2[s])
            want[s] = c.hmc_run(sampler, np.arange(K), boxes[s], **kw)
        finally:
            c.close()
    c = Context(0)
    try:
        _configure(c, F1, 0)
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        c.config_obs_periods(use)
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
                pos = np.concatenate([np.arange(nt), nt + np.flatnonzero(use[s])])
                assert np.array_equal(got["syn"][r][..., pos], want[s]["syn"], equal_nan=True), (resident, s)
                miss = nt + np.flatnonzero(~use[s])
                filled = np.abs(np.nan_to_num(got["syn"][r][..., :nt])).sum(axis=-1) > 0  # rows produced
                assert filled.any() and np.isnan(got["syn"][r][..., miss][filled]).all()
    finally:
        c.set_hmc_options(resident=0)
        c.close()


def _f1_joint():
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    cfg = f1_config()
    rf = ReceiverFunc(cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                      cfg["rf_type"], cfg["method"])
    return Joint_RF_SWD(1.0, 1.0, rf, SurfWD(tRc=T, tRg=T.copy()))


def test_station_array_with_periods_matches_its_station_models(tmp_path):
    from rfsurfhmc_b200.model.stations import StationArray
    from rfsurfhmc_b200.pyhmc.hmc import HamitonianMC
    from rfsurfhmc_b200.pyhmc.hmcda import HMCDualAveraging
    use = _masks(F1, 2, seed=8, no_rg=0)
    dobs = _stations(F1, 0, 2, seed=6)
    sa = StationArray(_f1_joint(), dobs, sigma1=[1.0, 0.5], names=["AA01", "BB02"], swd_use=use)
    X, _ = _rows(F1, B=16, seed=2, nsta=2)
    got = sa.misfit_and_grad_batch(X, np.arange(16) % 2)
    nt = _rf_len(0)
    for s in range(2):
        m = sa.station_model(s)
        assert np.array_equal(m.swdmodel.tRc, T[use[s][:36]]) and m.swdmodel.ntRg == use[s][36:].sum()
        b = m.misfit_and_grad_batch(X[s::2])
        for i in (0, 1, 3):
            assert np.array_equal(got[i][s::2], b[i])
        ok = b[3]
        pos = np.concatenate([np.arange(nt), nt + np.flatnonzero(use[s])])
        assert np.array_equal(got[2][s::2][ok][:, pos], b[2][ok])
        assert np.isnan(got[2][s::2][ok][:, nt + np.flatnonzero(~use[s])]).all()
    bounds = driver_bounds(f1_true_model())
    for cls, args in ((HamitonianMC, (0.1, (5, 20), 3, 991206, 4, 1)), (HMCDualAveraging, (0.02, 10, 3, 0.65, 991206, 4, 1))):
        hmc = cls(sa, bounds, *args, name="ch", outdir=str(tmp_path / cls.__name__))
        hmc.max_iters = 12
        out = hmc.sample_chains([0, 1, 0], stations=[0, 0, 1], save=True)
        one = cls(sa.station_model(1), bounds, *args, name="one", outdir=str(tmp_path / cls.__name__))
        one.max_iters = 12
        ref = one.sample_chains([0])
        for k in ("misfit", "samples", "n_iter", "n_acc"):
            assert np.array_equal(out[k][2], ref[k][0], equal_nan=True), (cls.__name__, k)
        f = np.load(tmp_path / cls.__name__ / "BB02" / "ch.0.npz")
        assert np.array_equal(f["obs"], dobs[1])
        assert f["syn"].shape[0] > 0 and np.isnan(f["syn"][:, nt + np.flatnonzero(~use[1])]).all()


def test_driver_runs_a_stations_file_with_periods(tmp_path):
    from rfsurfhmc_b200 import driver
    with open(os.path.join(ROOT, "tests", "golden", "f1_param.yaml")) as fh:
        param = yaml.safe_load(fh)
    dobs = _stations(F1, 0, 2, seed=7)
    use = _masks(F1, 2, seed=9, no_rg=1)

    def run(tag, **keys):
        param["hmc"].update(OUTPUT_DIR=str(tmp_path / tag), nsamples=3, ndraws=1)
        path = tmp_path / f"{tag}.npz"
        np.savez(path, **keys)
        return driver.run(param, "base", 2, save_chains=False, max_iters=8, stations=str(path))[0]

    both = run("both", dobs=dobs, names=np.array(["N1", "N2"]), swd_use=use)
    alone = run("alone", dobs=dobs[1:], names=np.array(["N2"]), swd_use=use[1:])
    grid = run("grid", dobs=dobs, names=np.array(["N1", "N2"]))
    assert np.array_equal(np.load(tmp_path / "both" / "N2" / "misfit.npy"), both[2:], equal_nan=True)
    assert np.isfinite(both).all() and np.array_equal(both[2:], alone)
    assert not np.array_equal(both[2:], grid[2:], equal_nan=True)


def test_joint_evaluator_with_obs_swd_use():
    from rfsurfhmc_b200.batched import JointEvaluator
    cfg = f1_config()
    cfg.update(sigma1=SIGMA1, sigma2=SIGMA2)
    use = _masks(F1, no_rg=4)
    dobs = _stations(F1, 0)
    X, sets = _rows(F1, B=128, seed=12)
    want, _, _ = _grouped(F1, 0, use, dobs, X, sets)
    ev = JointEvaluator(cfg, dobs, 7, obs_swd_use=use)
    dev = torch.device("cuda", 0)
    U, G, D, F = ev(torch.from_numpy(X).to(dev), torch.from_numpy(sets).to(dev))
    torch.cuda.synchronize(dev)
    got = [U.cpu().numpy(), G.cpu().numpy(), D.cpu().numpy(), F.cpu().numpy().astype(bool)]
    ev.ctx.close()
    _assert_same(got, want, "JointEvaluator")
