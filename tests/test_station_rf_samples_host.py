"""Per-station receiver-function samples, host side (no GPU): the stations-file key `rf_use`, the
rf_time_window helper and the checks and ray-subset models StationArray makes before it touches a
device."""
import numpy as np
import pytest
from rfsurfhmc_b200.fixtures import driver_bounds, f1_config, f1_true_model
from rfsurfhmc_b200.model.model_rf import ReceiverFunc
from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
from rfsurfhmc_b200.model.model_surf import SurfWD
from rfsurfhmc_b200.model.stations import StationArray, load_stations, rf_time_window, station_rf_samples

S, NP = 3, 14
T = np.arange(5., 41.)
RAYS = [0.04, 0.055, 0.07]


def _default():
    return driver_bounds(f1_true_model())


def _rf(rays=RAYS, nt=None, dt=None, time_shift=None):
    cfg = f1_config()
    return ReceiverFunc(rays, cfg["nt"] if nt is None else nt, cfg["dt"] if dt is None else dt, cfg["gauss"],
                        cfg["time_shift"] if time_shift is None else time_shift, cfg["water"], cfg["rf_type"],
                        cfg["method"])


def _joint(rf=None):
    return Joint_RF_SWD(1.0, 1.0, _rf() if rf is None else rf, SurfWD(tRc=T, tRg=T.copy()))


def _use(rf):
    u = np.ones((S, rf.nray, rf.nt_trace), dtype=bool)
    u[0, 1] = False      # station 0 misses the middle ray bin
    u[2, 0] = False      # station 2 misses the first two
    u[2, 1] = False
    return u


def test_station_rf_samples_accepts_both_shapes():
    rf = _rf()
    u = _use(rf)
    a = station_rf_samples(u, S, rf)
    b = station_rf_samples(u.reshape(S, -1).astype(np.int8), S, rf)
    assert a.dtype == bool and a.shape == (S, rf.nt) and np.array_equal(a, b)
    assert np.array_equal(a, u.reshape(S, -1))


@pytest.mark.parametrize("use,msg", [
    (np.ones((S, 3 * 125 - 1), dtype=bool), "shape"),    # wrong nray * nt
    (np.ones((S - 1, 3 * 125), dtype=bool), "shape"),    # wrong station count
    (np.ones((S, 125, 3), dtype=bool), "shape"),         # [S, nt, nray]
    (np.ones(3 * 125, dtype=bool), "shape"),
    (np.full((S, 3 * 125), 2), "0/1"),                    # not a mask
    (np.full((S, 3, 125), 0.5), "0/1"),
    (np.vstack((np.ones((S - 1, 375)), np.zeros((1, 375)))), "station 2 observes no receiver-function sample"),
])
def test_station_rf_samples_rejects_bad_masks_naming_the_key(use, msg):
    rf = _rf()
    with pytest.raises(ValueError, match=f"stations file: 'rf_use'.*{msg}"):
        station_rf_samples(use, S, rf, "stations file: ")
    nd = _joint().ndata
    with pytest.raises(ValueError, match=f"stations file: 'rf_use'.*{msg}"):
        load_stations({"dobs": np.zeros((S, nd)), "rf_use": use}, nd, NP, _default(), nray=3, rf=rf)


def test_loader_accepts_per_station_rf_samples_in_both_shapes(tmp_path):
    rf = _rf()
    nd = _joint().ndata
    dobs = np.zeros((S, nd))
    assert load_stations({"dobs": dobs}, nd, NP, _default(), nray=3, rf=rf)["rf_use"] is None
    for k, u in enumerate((_use(rf), _use(rf).reshape(S, -1))):
        path = tmp_path / f"st{k}.npz"
        np.savez(path, dobs=dobs, rf_use=u.astype(np.uint8))
        st = load_stations(str(path), nd, NP, _default(), nray=3, rf=rf)
        assert st["rf_use"].dtype == bool and np.array_equal(st["rf_use"], _use(rf).reshape(S, -1))


def test_loader_needs_an_rf_configuration_for_the_mask():
    with pytest.raises(ValueError, match="'rf_use'.*receiver-function configuration"):
        load_stations({"dobs": np.zeros((S, 72)), "rf_use": np.ones((S, 125))}, 72, NP, _default())


def test_rf_time_window_edges_on_samples():
    # dt = 0.25 and time_shift = 2 are exact in binary: t = -2, -1.75, ..., every bound lands on a sample
    rf = _rf(rays=[0.05, 0.06], nt=64, dt=0.25, time_shift=2.0)
    assert rf.t[0] == -2.0 and rf.t[8] == 0.0
    u = rf_time_window(rf, [-2.0, 0.0, -1.0], [15.75, 1.0, 0.0])
    assert u.shape == (S, 2 * 64) and u.dtype == bool
    u = u.reshape(S, 2, 64)
    assert u[0].all()                                     # the whole trace, both bounds on the end samples
    assert np.array_equal(np.flatnonzero(u[1, 0]), np.arange(8, 13))   # 0 s .. 1 s inclusive
    assert np.array_equal(np.flatnonzero(u[2, 1]), np.arange(4, 9))    # -1 s .. 0 s inclusive
    assert np.array_equal(u[:, 0], u[:, 1])               # [S] bounds apply to every ray


def test_rf_time_window_bounds_written_in_seconds_survive_rounding():
    # dt = 0.4, time_shift = 5 (F1): k * 0.4 - 5 is not exact, yet a bound written as a sample time selects it
    rf = _rf(rays=0.045)
    assert rf.t[17] > 1.8  # 1.8000000000000007
    u = rf_time_window(rf, [0.2], [1.8])[0]
    assert np.array_equal(np.flatnonzero(u), np.arange(13, 18))


def test_rf_time_window_per_ray_bounds_and_missing_rays():
    rf = _rf(rays=[0.05, 0.06, 0.07], nt=64, dt=0.25, time_shift=2.0)
    lo = np.array([[-2.0, np.nan, 0.0], [0.0, 0.0, 0.0], [np.nan, -1.0, np.nan]])
    hi = np.array([[1.0, 3.0, np.nan], [5.0, 10.0, 15.75], [2.0, 2.0, 2.0]])
    u = rf_time_window(rf, lo, hi).reshape(S, 3, 64)
    assert np.array_equal(np.flatnonzero(u[0, 0]), np.arange(0, 13))
    assert not u[0, 1].any() and not u[0, 2].any()        # NaN in either bound: ray not observed
    assert np.array_equal(np.flatnonzero(u[1, 2]), np.arange(8, 64))
    assert [int(r.sum()) for r in u[1]] == [21, 41, 56]
    assert not u[2, 0].any() and np.array_equal(np.flatnonzero(u[2, 1]), np.arange(4, 17)) and not u[2, 2].any()
    with pytest.raises(ValueError, match=r"\[S\] or \[S, 3\]"):
        rf_time_window(rf, lo[:, :2], hi[:, :2])
    with pytest.raises(ValueError, match=r"\[S\] or \[S, 3\]"):
        rf_time_window(rf, lo, hi[:, 0])
    # the mask feeds StationArray as it is
    sa = StationArray(rf, np.zeros((S, rf.nt)), rf_use=rf_time_window(rf, lo, hi))
    assert np.array_equal(sa.rf_use, u.reshape(S, -1))


def test_station_array_validates_rf_masks_before_any_device():
    joint = _joint()
    dobs = np.zeros((S, joint.ndata))
    u = _use(joint.rfmodel)
    sa = StationArray(joint, dobs, rf_use=u)
    assert sa.rf_use.dtype == bool and sa.rf_use.shape == (S, 375) and sa._ctx is None
    assert StationArray(joint, dobs).rf_use is None
    for bad in (u[:, 1:], u[1:], np.full((S, 375), 3)):
        with pytest.raises(ValueError, match="'rf_use'"):
            StationArray(joint, dobs, rf_use=bad)
    v = u.copy()
    v[1] = False
    with pytest.raises(ValueError, match="station 1 observes no receiver-function sample"):
        StationArray(joint, dobs, rf_use=v)
    swd = SurfWD(tRc=T, tRg=T.copy())
    with pytest.raises(TypeError, match="rf_use"):
        StationArray(swd, np.zeros((S, swd.nt)), rf_use=np.ones((S, 375), dtype=bool))
    rf = _rf()
    assert StationArray(rf, np.zeros((S, rf.nt)), rf_use=u.astype(int)).rf_use.shape == (S, 375)


def test_station_model_keeps_the_observed_rays():
    joint = _joint()
    nt = 125
    dobs = np.arange(S * joint.ndata, dtype=np.float64).reshape(S, joint.ndata)
    p = np.array([[0.041, 0.052, 0.063], [0.042, 0.053, 0.064], [0.043, 0.054, 0.065]])
    sa = StationArray(joint, dobs, rf_use=_use(joint.rfmodel), ray_p=p, names=["A", "B", "C"])
    m = sa.station_model(0)
    assert m.rfmodel.ray_p == [0.041, 0.063] and m.rfmodel.nray == 2 and m.rfmodel.nt == 2 * nt
    assert m.ndata == 2 * nt + 72
    assert np.array_equal(m.dobs, np.concatenate((dobs[0, :nt], dobs[0, 2 * nt:])))
    m = sa.station_model(1)
    assert m.rfmodel.ray_p == p[1].tolist() and m.rfmodel.nt == 3 * nt and np.array_equal(m.dobs, dobs[1])
    m = sa.station_model(2)
    assert m.rfmodel.ray_p == 0.065 and m.rfmodel.nray == 1 and m.rfmodel.nt == nt
    assert np.array_equal(m.dobs, dobs[2, 2 * nt:])
    # the template keeps its rays; without a ray table the template's values are subset
    assert joint.rfmodel.ray_p == RAYS and joint.rfmodel.nt == 3 * nt
    m = StationArray(joint, dobs, rf_use=_use(joint.rfmodel)).station_model(0)
    assert m.rfmodel.ray_p == [RAYS[0], RAYS[2]]
    # an RF-only template
    rf = _rf()
    d = np.arange(S * rf.nt, dtype=np.float64).reshape(S, rf.nt)
    m = StationArray(rf, d, rf_use=_use(rf)).station_model(2)
    assert m.ray_p == RAYS[2] and m.nt == nt and np.array_equal(m.dobs, d[2, 2 * nt:])


def test_station_model_refuses_a_partial_window():
    joint = _joint()
    u = _use(joint.rfmodel)
    u[1, 2, 100:] = False  # station 1 cuts its last ray's coda
    sa = StationArray(joint, np.zeros((S, joint.ndata)), rf_use=u, names=["A", "B", "C"])
    sa.station_model(0)
    with pytest.raises(ValueError, match=r"station 1 \(B\) fits part of a receiver-function trace"):
        sa.station_model(1)
    assert sa.station_view(1).dobs.shape == (joint.ndata,)
