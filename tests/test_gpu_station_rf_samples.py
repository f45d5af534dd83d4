"""Per-station receiver-function samples (rfs_config_obs_rf_samples).  A station that misses whole ray
bins must give exactly what a context holding only that station, configured through config_rf on its
observed rays, gives, in grouped evaluations and in the grouped HMC.  A station that fits part of a trace
must give exactly what an unmasked context gives when dobs at its unobserved samples is replaced by the
row's own synthetic (the residual there is then exactly 0).  dsyn keeps the full traces."""
import os
import ctypes
import numpy as np
import pytest
import torch
import yaml
from rfsurfhmc_b200._lib import Context, RfsError
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models
from rfsurfhmc_b200.pyhmc._common import chain_status

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RFS_E_ARG, RFS_E_CONFIG = -2, -4
S = 5
SIGMA1 = np.array([1.0, 0.5, 2.0, 1.0, 0.8])
SIGMA2 = np.array([1.0, 1.5, 1.0, 0.25, 1.0])
RAYS = [0.04, 0.055, 0.07]
TABLE = np.array([[0.041, 0.052, 0.066], [0.043, 0.057, 0.071], [0.045, 0.054, 0.068], [0.039, 0.058, 0.073],
                  [0.044, 0.056, 0.069]])
NT = f1_config()["nt"]
NR = len(RAYS)
NRF = NR * NT
NSW = 72
T = np.arange(5., 41.)
METHODS = ["freq", "time"]


def _configure(c, which, method="freq", rays=RAYS, lists=None):
    cfg = f1_config()
    if which != 1:
        c.config_swd(7, *((T, T.copy()) if lists is None else lists))
    if which != 2:
        c.config_rf(7, rays, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], cfg["rf_type"],
                    method)


def _stations(which, method, nsta=S, seed=3, table=None):
    """Observations of nsta stations: seeded perturbations of the F1 true model plus seeded noise."""
    c = Context(0)
    try:
        _configure(c, which, method)
        c.config_obs(np.zeros((nsta, c.ndata(which))))
        if table is not None:
            c.config_obs_rays(table[:nsta])
        _, _, d, _ = c.misfit_grad_host(perturbed_models(f1_true_model(), nsta, seed=seed, rel=0.05), which,
                                        sets=np.arange(nsta))
    finally:
        c.close()
    d = np.where(np.isfinite(d), d, 0.0)
    return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)


def _rows(B=333, seed=8, nsta=S):
    """Models near the truth, strongly perturbed ones and ones with a slow half-space (many of those fail
    the SWD root search), each row on a random station; every station appears."""
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


def _whole(nsta=S):
    """Whole-trace masks [nsta, NRF]: station 1 misses the middle bin, 2 the first two, 3 the last, 4 the
    first."""
    obs = np.ones((S, NR), dtype=bool)
    obs[1, 1] = obs[2, 0] = obs[2, 1] = obs[3, 2] = obs[4, 0] = False
    return np.repeat(obs[:nsta], NT, axis=1)


def _windows(nsta=S, seed=1):
    """Partial windows [nsta, NRF]: every trace a seeded window of 40-100 % of its samples; station 3
    misses the middle bin."""
    rng = np.random.default_rng(seed)
    u = np.zeros((nsta, NR, NT), dtype=bool)
    for s in range(nsta):
        for r in range(NR):
            k = int(rng.integers(int(np.ceil(0.4 * NT)), NT + 1))
            a = int(rng.integers(0, NT - k + 1))
            u[s, r, a:a + k] = True
    if nsta > 3:
        u[3, 1] = False
    return u.reshape(nsta, NRF)


def _swd_masks(nsta=S, seed=4):
    rng = np.random.default_rng(seed)
    u = np.ones((nsta, NSW), dtype=bool)
    for s in range(nsta):
        for o in (0, 36):
            k = int(rng.integers(22, 37))
            a = int(rng.integers(0, 36 - k + 1))
            u[s, o:o + 36] = False
            u[s, o + a:o + a + k] = True
    return u


def _grouped(which, method, dobs, X, sets, use=None, table=None, swd_use=None, ctx=None):
    c = Context(0) if ctx is None else ctx
    try:
        _configure(c, which, method)
        c.config_obs(dobs, SIGMA1[:len(dobs)], SIGMA2[:len(dobs)])
        if table is not None:
            c.config_obs_rays(table[:len(dobs)])
        if swd_use is not None:
            c.config_obs_periods(swd_use)
        if use is not None:
            c.config_obs_rf_samples(use)
        return c.misfit_grad_host(X, which, sets=sets)
    finally:
        if ctx is None:
            c.close()


def _per_station(which, method, use, dobs, X, sets, table=None, swd_use=None):
    """Reference: one context per station on its observed rays (and periods); U, grad, flag per row and
    dsyn at the station's observed data positions."""
    out = [np.zeros(len(X)), np.zeros(X.shape), [None] * len(X), np.zeros(len(X), dtype=bool)]
    for s in range(len(dobs)):
        r = np.flatnonzero(sets == s)
        if r.size == 0:
            continue
        obs = use[s].reshape(NR, NT).all(axis=1)
        rays = (np.asarray(RAYS) if table is None else table[s])[obs]
        pos = np.flatnonzero(use[s])
        lists = None
        if which != 1 and swd_use is not None:
            lists = (T[swd_use[s][:36]], T[swd_use[s][36:]])
            pos = np.concatenate((pos, NRF + np.flatnonzero(swd_use[s])))
        elif which != 1:
            pos = np.concatenate((pos, NRF + np.arange(NSW)))
        c = Context(0)
        try:
            _configure(c, which, method, rays.tolist(), lists)
            c.config_obs(dobs[s][pos], SIGMA1[s], SIGMA2[s])
            U, g, d, f = c.misfit_grad_host(X[r], which)
        finally:
            c.close()
        out[0][r], out[1][r], out[3][r] = U, g, f
        for i, b in enumerate(r):
            out[2][b] = (pos, d[i])
    return out


def _assert_per_station(got, want, tag):
    for name, i in (("U", 0), ("grad", 1), ("flag", 3)):
        assert np.array_equal(got[i], want[i]), (tag, name)
    for b, (pos, d) in enumerate(want[2]):
        assert np.array_equal(got[2][b][pos], d, equal_nan=True), (tag, "dsyn", b)


def _assert_same(got, want, tag, rows=slice(None)):
    for name, a, b in zip(("U", "grad", "dsyn", "flag"), got, want):
        assert np.array_equal(a[rows], b[rows], equal_nan=True), (tag, name)


# (name, which, method, per-station ray table, period mask)
WHOLE = [(f"{'joint' if w == 0 else 'rf'}_{m}", w, m, None, False) for w in (0, 1) for m in METHODS] + [
    ("joint_freq_ray_table", 0, "freq", TABLE, False),
    ("rf_time_ray_table", 1, "time", TABLE, False),
    ("joint_freq_periods", 0, "freq", None, True),
    ("joint_time_periods_ray_table", 0, "time", TABLE, True),
]


@pytest.mark.parametrize("name,which,method,table,periods", WHOLE, ids=[c[0] for c in WHOLE])
def test_whole_trace_masks_equal_per_station_ray_subsets(name, which, method, table, periods):
    use = _whole()
    dobs = _stations(which, method, table=table)
    X, sets = _rows()
    swd_use = _swd_masks() if periods else None
    got = _grouped(which, method, dobs, X, sets, use, table, swd_use)
    want = _per_station(which, method, use, dobs, X, sets, table, swd_use)
    _assert_per_station(got, want, name)
    # dsyn keeps the full traces: the unobserved rays are the synthetics of the unmasked context
    plain = _grouped(which, method, dobs, X, sets, None, table, swd_use)
    ok = got[3]
    assert np.array_equal(got[2][ok][:, :NRF], plain[2][ok][:, :NRF])
    assert np.isfinite(got[2][ok][:, :NRF]).all()
    if which == 0:
        fail = ~got[3]
        assert fail.any() and fail.sum() < len(X) // 2
        assert np.array_equal(got[2][fail], dobs[sets[fail]])  # the failure convention: the station's dobs
        assert not np.array_equal(got[0][ok], plain[0][ok])


def _substituted(which, method, use, dobs, X, sets):
    """Comparison for partial windows: an unmasked context with one set per row whose dobs holds the
    station's values at observed samples and the row's own synthetic (from an unmasked evaluation) at
    the others."""
    syn = _grouped(1, method, dobs[:, :NRF], X, sets)[2]
    d = dobs[sets].copy()
    m = use[sets]
    d[:, :NRF][~m] = syn[~m]
    c = Context(0)
    try:
        _configure(c, which, method)
        c.config_obs(d, SIGMA1[sets], SIGMA2[sets])
        return c.misfit_grad_host(X, which, sets=np.arange(len(X), dtype=np.int32))
    finally:
        c.close()


@pytest.mark.parametrize("method", METHODS)
def test_partial_windows_rf_only_equal_a_substitution(method):
    use = _windows()
    dobs = _stations(1, method)
    X, sets = _rows(B=200, seed=6)
    got = _grouped(1, method, dobs, X, sets, use)
    want = _substituted(1, method, use, dobs, X, sets)
    for name, i in (("U", 0), ("grad", 1), ("flag", 3)):
        assert np.array_equal(got[i], want[i]), (method, name)
    assert np.array_equal(got[2], _grouped(1, method, dobs, X, sets)[2])  # full traces
    assert not np.array_equal(got[0], _grouped(1, method, dobs, X, sets)[0])


@pytest.mark.parametrize("method", METHODS)
def test_partial_windows_joint_weight_uses_each_sets_sample_count(method):
    use = _windows()
    dobs = _stations(0, method)
    X, sets = _rows(B=200, seed=7)
    got = _grouped(0, method, dobs, X, sets, use)
    rf = _grouped(1, method, dobs[:, :NRF], X, sets, use)
    sw = _grouped(2, method, dobs[:, NRF:], X, sets)
    n1 = use.sum(axis=1)
    assert len(set(n1.tolist())) == S
    wt = (SIGMA1 / SIGMA2) ** 2 * n1 / NSW
    ok = got[3]
    assert ok.sum() > len(X) // 2 and np.array_equal(ok, sw[3])
    w = wt[sets[ok]]
    U = rf[0][ok] + w * sw[0][ok]
    G = rf[1][ok] + w[:, None] * sw[1][ok]
    assert np.all(np.abs(got[0][ok] - U) <= 1e-12 * np.abs(U))
    assert np.all(np.abs(got[1][ok] - G) <= 1e-12 * np.abs(G).max(axis=1, keepdims=True))
    assert np.array_equal(got[2][ok][:, :NRF], rf[2][ok])


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("method", METHODS)
def test_all_ones_mask_gives_the_bits_of_no_table(which, method):
    dobs = _stations(which, method)
    X, sets = _rows(B=160, seed=11)
    want = _grouped(which, method, dobs, X, sets)
    got = _grouped(which, method, dobs, X, sets, np.ones((S, NR, NT), dtype=np.uint8))
    _assert_same(got, want, "all ones")


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("method", METHODS)
def test_values_at_unobserved_samples_are_never_read(which, method):
    use = _windows(seed=5)
    dobs = _stations(which, method)
    X, sets = _rows(B=160, seed=12)
    outs = []
    for fill in (0.0, np.nan, 1e300, -1e300):
        d = dobs.copy()
        d[:, :NRF][~use] = fill
        outs.append(_grouped(which, method, d, X, sets, use))
    for o in outs[1:]:
        for i in (0, 1, 3):
            assert np.array_equal(o[i], outs[0][i])
        ok = outs[0][3]
        assert np.array_equal(o[2][ok], outs[0][2][ok])  # a failed row returns its own dobs
    assert np.isfinite(outs[1][0]).all() and np.isfinite(outs[1][1]).all()


def _raw(c, S_, use):
    if use is None:
        return c.L.rfs_config_obs_rf_samples(c.h, S_, NRF, None)
    u = np.ascontiguousarray(use, dtype=np.uint8)
    return c.L.rfs_config_obs_rf_samples(c.h, S_, u.shape[1], u.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)))


def test_config_obs_rf_samples_errors():
    use = _windows()
    c = Context(0)
    try:
        _configure(c, 2)  # SWD only: no RF configuration
        c.config_obs(np.zeros((S, c.ndata(2))))
        with pytest.raises(RfsError) as e:
            c.config_obs_rf_samples(use)
        assert e.value.code == RFS_E_CONFIG
    finally:
        c.close()
    dobs = _stations(0, "freq")
    X, sets = _rows(B=64, seed=9)
    c = Context(0)
    try:
        _configure(c, 0)
        with pytest.raises(RfsError) as e:  # no observation sets yet
            c.config_obs_rf_samples(use)
        assert e.value.code == RFS_E_CONFIG
        c.config_obs(dobs, SIGMA1, SIGMA2)
        plain = c.misfit_grad_host(X, 0, sets=sets)
        with pytest.raises(RfsError) as e:  # S differs from the sets held
            c.config_obs_rf_samples(use[:S - 1])
        assert e.value.code == RFS_E_CONFIG
        with pytest.raises(RfsError) as e:  # wrong nrf
            c.config_obs_rf_samples(use[:, 1:])
        assert e.value.code == RFS_E_ARG
        assert _raw(c, S, None) == RFS_E_ARG
        bad = use.astype(np.uint8)
        bad[2, 40] = 2
        assert _raw(c, S, bad) == RFS_E_ARG
        bad = use.copy()
        bad[3] = False
        with pytest.raises(RfsError) as e:  # a station fitting no sample
            c.config_obs_rf_samples(bad)
        assert e.value.code == RFS_E_ARG
        # a failed call leaves no table, also after a valid one
        c.config_obs_rf_samples(use)
        masked = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(masked[0], plain[0])
        assert _raw(c, S, bad) == RFS_E_ARG
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "failed call")
        c.config_obs_rf_samples(use)
        with pytest.raises(RfsError):
            c.config_obs_rf_samples(use[:S - 1])
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "failed call (config)")
    finally:
        c.close()


def test_config_calls_drop_or_keep_the_table():
    """rfs_config_obs_sets, rfs_config_obs, rfs_config_rf and rfs_config_rf_rays drop the table;
    rfs_config_swd, rfs_config_obs_rays and rfs_config_obs_periods keep it; which = 2 ignores it."""
    cfg = f1_config()
    use = _windows(seed=2)
    dobs = _stations(0, "freq")
    X, sets = _rows(B=96, seed=10)
    c = Context(0)
    try:
        _configure(c, 0)
        c.config_obs(dobs, SIGMA1, SIGMA2)
        plain = c.misfit_grad_host(X, 0, sets=sets)
        c.config_obs_rf_samples(use)
        masked = c.misfit_grad_host(X, 0, sets=sets)
        assert not np.array_equal(masked[0], plain[0])
        sw = Context(0)
        try:  # which = 2 ignores the table (the context holds SWD data only, but an RF configuration too)
            _configure(sw, 0)
            sw.config_obs(dobs[:, NRF:], SIGMA1, SIGMA2)
            swd_plain = sw.misfit_grad_host(X, 2, sets=sets)
            sw.config_obs_rf_samples(use)
            _assert_same(sw.misfit_grad_host(X, 2, sets=sets), swd_plain, "which = 2 ignores the table")
        finally:
            sw.close()
        # kept
        c.config_swd(7, T, T.copy())
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), masked, "config_swd keeps")
        c.config_obs_rays(np.tile(RAYS, (S, 1)))  # a table of the shared values: the bits of none
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), masked, "config_obs_rays keeps")
        c.config_obs_periods(np.ones((S, NSW), dtype=bool))
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), masked, "config_obs_periods keeps")
        # dropped
        c.config_obs(dobs, SIGMA1, SIGMA2)  # rfs_config_obs_sets
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "config_obs_sets")
        c.config_obs_rf_samples(use)
        _configure(c, 1)  # rfs_config_rf_rays
        _assert_same(c.misfit_grad_host(X, 0, sets=sets), plain, "config_rf_rays")
        one = Context(0)
        try:  # rfs_config_rf (the scalar call) on a one-ray context
            _configure(one, 1, rays=RAYS[0])
            one.config_obs(dobs[:, :NT])
            one_plain = one.misfit_grad_host(X, 1, sets=sets)
            one.config_obs_rf_samples(use[:, :NT] | ~use[:, :NT].any(axis=1, keepdims=True))
            assert not np.array_equal(one.misfit_grad_host(X, 1, sets=sets)[0], one_plain[0])
            assert one.L.rfs_config_rf(one.h, 7, ctypes.c_double(RAYS[0]), cfg["nt"], cfg["dt"], cfg["gauss"],
                                       cfg["time_shift"], cfg["water"], 1, 1) == 0
            _assert_same(one.misfit_grad_host(X, 1, sets=sets), one_plain, "config_rf")
        finally:
            one.close()
        # rfs_config_obs (the one-set call)
        r = sets == 2
        c.config_obs(dobs[2], SIGMA1[2], SIGMA2[2])
        want = c.misfit_grad_host(X[r], 0)
        c.config_obs_rf_samples(use[2:3])
        assert np.array_equal(c.misfit_grad_host(X[r], 0)[0], masked[0][r])
        d2 = np.ascontiguousarray(dobs[2])
        assert c.L.rfs_config_obs(c.h, SIGMA1[2], SIGMA2[2], d2.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                  d2.size) == 0
        _assert_same(c.misfit_grad_host(X[r], 0), want, "config_obs")
    finally:
        c.close()


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
    use = _windows(seed=3)
    dobs = _stations(which, method)
    X, sets = _rows(B=96, seed=4)
    c = Context(0)
    try:
        want = _grouped(which, method, dobs, X, sets, use, ctx=c)
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


@pytest.mark.parametrize("which,method", [(0, "freq"), (1, "time")])
def test_chunked_batch_uses_each_rows_own_mask(which, method):
    """A 1 MiB workspace budget forces many 32-row chunks: each chunk's residual kernels must read the
    masks of its own rows."""
    use = _windows(seed=6)
    dobs = _stations(which, method)
    X, sets = _rows()
    plain = Context(0)
    try:
        n0 = plain.launches
        want = _grouped(which, method, dobs, X, sets, use, ctx=plain)
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
        got = _grouped(which, method, dobs, X, sets, use, ctx=c)
        assert c.launches - n0 >= 4 * plain_launches  # really chunked
    finally:
        c.close()
    _assert_same(got, want, "chunked")


def _boxes(nsta):
    b = np.repeat(driver_bounds(f1_true_model())[None], nsta, axis=0)
    for s in range(nsta):
        b[s, :7, 0] *= 1.0 + 0.04 * s
        b[s, :7, 1] *= 1.0 - 0.03 * s
    return b


def _hmc_kw(sampler):
    kw = (dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=6, ndraws=1, max_iters=14) if sampler == 0 else
          dict(dt=0.02, L0=10, target_ratio=0.65, seed=991206, nsamples=3, ndraws=3, max_iters=14))
    kw.update(want_samples=True, want_syn=True, log_accepts=kw["max_iters"])
    return kw


@pytest.mark.parametrize("sampler", [0, 1])
def test_hmc_with_whole_trace_masks_equals_single_station_runs(sampler):
    nsta, K = 3, 6
    kw = _hmc_kw(sampler)
    boxes = _boxes(nsta)
    use = _whole(nsta)
    dobs = _stations(0, "freq", nsta, seed=5)
    want = {}
    for s in range(nsta):
        obs = use[s].reshape(NR, NT).all(axis=1)
        pos = np.concatenate((np.flatnonzero(use[s]), NRF + np.arange(NSW)))
        c = Context(0)
        try:
            _configure(c, 0, rays=np.asarray(RAYS)[obs].tolist())
            c.config_obs(dobs[s][pos], SIGMA1[s], SIGMA2[s])
            want[s] = c.hmc_run(sampler, np.arange(K), boxes[s], **kw)
        finally:
            c.close()
    c = Context(0)
    try:
        _configure(c, 0)
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        c.config_obs_rf_samples(use)
        ids = np.tile(np.arange(K), nsta)
        sets = np.repeat(np.arange(nsta), K)
        got = c.hmc_run(sampler, ids, boxes, sets=sets, **kw)
        assert len(set(got["n_iter"].tolist())) > 1  # chains finish at different steps: compaction
        for s in range(nsta):
            r = sets == s
            for k in ("samples", "misfit", "n_iter", "n_acc", "accept_seq", "initmodel", "dt"):
                assert np.array_equal(got[k][r], want[s][k], equal_nan=True), (s, k)
            pos = np.concatenate((np.flatnonzero(use[s]), NRF + np.arange(NSW)))
            assert np.array_equal(got["syn"][r][..., pos], want[s]["syn"], equal_nan=True), s
    finally:
        c.close()


@pytest.mark.parametrize("sampler", [0, 1])
def test_hmc_with_partial_windows_is_the_same_with_resident_slots(sampler):
    nsta, K = 4, 5
    kw = _hmc_kw(sampler)
    boxes = _boxes(nsta)
    use = _windows(nsta, seed=8)
    dobs = _stations(0, "freq", nsta, seed=6)
    c = Context(0)
    try:
        _configure(c, 0)
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        c.config_obs_rf_samples(use)
        ids = np.tile(np.arange(K), nsta)
        sets = np.repeat(np.arange(nsta), K)
        outs = []
        for resident in (0, 7):
            c.set_hmc_options(resident=resident)
            outs.append(c.hmc_run(sampler, ids, boxes, sets=sets, **kw))
        for k in ("samples", "misfit", "n_iter", "n_acc", "accept_seq", "initmodel", "dt", "syn"):
            assert np.array_equal(outs[0][k], outs[1][k], equal_nan=True), k
        nv, _ = chain_status(outs[0], kw["nsamples"], kw["ndraws"])
        for i in range(len(ids)):
            assert np.isfinite(outs[0]["misfit"][i][:nv[i]]).all()
        assert nv.sum() > 0
        c.config_obs(dobs, SIGMA1[:nsta], SIGMA2[:nsta])
        plain = c.hmc_run(sampler, ids, boxes, sets=sets, **kw)
        assert not np.array_equal(plain["misfit"], outs[0]["misfit"], equal_nan=True)
    finally:
        c.set_hmc_options(resident=0)
        c.close()


def _f1_joint(method="freq"):
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    cfg = f1_config()
    rf = ReceiverFunc(RAYS, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], cfg["rf_type"],
                      method)
    return Joint_RF_SWD(1.0, 1.0, rf, SurfWD(tRc=T, tRg=T.copy()))


def test_station_array_with_rf_samples_matches_its_station_models(tmp_path):
    from rfsurfhmc_b200.model.stations import StationArray, rf_time_window
    from rfsurfhmc_b200.pyhmc.hmc import HamitonianMC
    nsta = 3
    use = _whole(nsta)
    dobs = _stations(0, "freq", nsta, seed=6)
    sa = StationArray(_f1_joint(), dobs, sigma1=SIGMA1[:nsta], names=["AA01", "BB02", "CC03"],
                      ray_p=TABLE[:nsta], rf_use=use.reshape(nsta, NR, NT))
    X, _ = _rows(B=18, seed=2, nsta=nsta)
    st = np.arange(18) % nsta
    got = sa.misfit_and_grad_batch(X, st)
    for s in range(nsta):
        m = sa.station_model(s)
        assert m.rfmodel.nray == use[s].reshape(NR, NT).all(axis=1).sum()
        b = m.misfit_and_grad_batch(X[st == s])
        for i in (0, 1, 3):
            assert np.array_equal(got[i][st == s], b[i])
        pos = np.concatenate((np.flatnonzero(use[s]), NRF + np.arange(NSW)))
        assert np.array_equal(got[2][st == s][:, pos], b[2])
    bounds = driver_bounds(f1_true_model())
    hmc = HamitonianMC(sa, bounds, 0.1, (5, 20), 3, 991206, 4, 1, name="ch", outdir=str(tmp_path))
    hmc.max_iters = 12
    out = hmc.sample_chains([0, 1, 0], stations=[0, 0, 2], save=True)
    one = HamitonianMC(sa.station_model(2), bounds, 0.1, (5, 20), 3, 991206, 4, 1, name="one", outdir=str(tmp_path))
    one.max_iters = 12
    ref = one.sample_chains([0])
    for k in ("misfit", "samples", "n_iter", "n_acc"):
        assert np.array_equal(out[k][2], ref[k][0], equal_nan=True), k
    f = np.load(tmp_path / "CC03" / "ch.0.npz")  # the array's data layout, full traces
    assert np.array_equal(f["obs"], dobs[2]) and f["syn"].shape[1] == NRF + NSW
    # a partial window: no station model, the grouped view still evaluates it
    win = rf_time_window(sa.template.rfmodel, [-2.2, -5.0, 0.2], [15.0, 20.0, 8.2])
    sw = StationArray(_f1_joint(), dobs, rf_use=win)
    with pytest.raises(ValueError, match="station 0"):
        sw.station_model(0)
    v = sw.station_view(0).misfit_and_grad(X[0])
    assert np.isfinite(v[0]) and v[2].shape == (NRF + NSW,)


def test_driver_runs_a_stations_file_with_rf_samples(tmp_path):
    from rfsurfhmc_b200 import driver
    with open(os.path.join(ROOT, "tests", "golden", "f1_param.yaml")) as fh:
        param = yaml.safe_load(fh)
    nt = param["rf"]["nt"]
    c = Context(0)
    try:
        _configure(c, 0, rays=param["rf"]["ray_p"])
        c.config_obs(np.zeros((2, c.ndata(0))))
        d = c.misfit_grad_host(perturbed_models(f1_true_model(), 2, seed=7, rel=0.05), 0, sets=np.arange(2))[2]
    finally:
        c.close()
    dobs = np.where(np.isfinite(d), d, 0.0)
    use = np.ones((2, 1, nt), dtype=bool)
    use[0, 0, :10] = use[1, 0, 60:] = False

    def run(tag, **keys):
        param["hmc"].update(OUTPUT_DIR=str(tmp_path / tag), nsamples=3, ndraws=1)
        path = tmp_path / f"{tag}.npz"
        np.savez(path, **keys)
        return driver.run(param, "base", 2, save_chains=True, max_iters=8, stations=str(path))[0]

    both = run("both", dobs=dobs, names=np.array(["N1", "N2"]), rf_use=use)
    alone = run("alone", dobs=dobs[1:], names=np.array(["N2"]), rf_use=use[1:].reshape(1, nt))
    full = run("full", dobs=dobs, names=np.array(["N1", "N2"]))
    assert np.array_equal(np.load(tmp_path / "both" / "N2" / "misfit.npy"), both[2:], equal_nan=True)
    assert np.array_equal(both[2:], alone, equal_nan=True)
    assert not np.array_equal(both[2:], full[2:], equal_nan=True)


def test_joint_evaluator_with_obs_rf_use():
    from rfsurfhmc_b200.batched import JointEvaluator
    cfg = f1_config()
    cfg.update(sigma1=SIGMA1, sigma2=SIGMA2, ray_p=RAYS)
    use = _windows(seed=9)
    dobs = _stations(0, "freq")
    X, sets = _rows(B=128, seed=12)
    want = _grouped(0, "freq", dobs, X, sets, use)
    ev = JointEvaluator(cfg, dobs, 7, obs_rf_use=use)
    dev = torch.device("cuda", 0)
    U, G, D, F = ev(torch.from_numpy(X).to(dev), torch.from_numpy(sets).to(dev))
    torch.cuda.synchronize(dev)
    got = [U.cpu().numpy(), G.cpu().numpy(), D.cpu().numpy(), F.cpu().numpy().astype(bool)]
    ev.ctx.close()
    _assert_same(got, want, "JointEvaluator")
