"""Gaussian-width lists, host side (no GPU): the data counts of ReceiverFunc and the shapes and checks of
the station helpers for the [ray][gauss][nt] layout of the receiver-function data."""
import numpy as np
import pytest
from rfsurfhmc_b200.fixtures import driver_bounds, f1_config, f1_true_model
from rfsurfhmc_b200.model.model_rf import ReceiverFunc
from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
from rfsurfhmc_b200.model.model_surf import SurfWD
from rfsurfhmc_b200.model.stations import StationArray, load_stations, rf_time_window, station_rf_samples

S, NP = 3, 14
T = np.arange(5., 41.)
RAYS = [0.04, 0.06]
WIDTHS = [1.0, 2.5, 5.0]
CFG = f1_config()
NT = CFG["nt"]


def _rf(rays=RAYS, gauss=WIDTHS):
    return ReceiverFunc(rays, NT, CFG["dt"], gauss, CFG["time_shift"], CFG["water"], CFG["rf_type"], CFG["method"])


def _joint(rf=None):
    return Joint_RF_SWD(1.0, 1.0, _rf() if rf is None else rf, SurfWD(tRc=T, tRg=T.copy()))


def test_receiver_func_counts_every_trace():
    rf = _rf()
    assert (rf.nray, rf.ngauss, rf.nt_trace, rf.nt) == (2, 3, NT, 2 * 3 * NT)
    assert _rf(0.045, 1.5).nt == NT and _rf(0.045, [1.5]).nt == NT and _rf(0.045, [1.0, 2.0]).nt == 2 * NT
    assert _joint().ndata == 6 * NT + 72
    # the widths are part of the configuration key: changing one re-configures the device context
    a = _rf()._config_fields(7)
    b = _rf(gauss=[1.0, 2.5, 4.0])._config_fields(7)
    assert a != b and _rf(gauss=1.5)._config_fields(7)[4] == 1.5
    rf = _rf(gauss=list(WIDTHS))
    key = rf._config_fields(7)
    rf.gauss[2] = 4.0           # an in-place change of the list is seen too
    assert rf._config_fields(7) != key


def test_station_rf_samples_shapes():
    rf = _rf()
    u = np.ones((S, 2, 3, NT), dtype=bool)
    u[0, 1, 2] = False
    a = station_rf_samples(u, S, rf)
    b = station_rf_samples(u.reshape(S, -1).astype(np.int8), S, rf)
    assert a.shape == (S, rf.nt) and a.dtype == bool and np.array_equal(a, b) and np.array_equal(a, u.reshape(S, -1))
    # [S, nray, nt] only with one width
    with pytest.raises(ValueError, match=r"'rf_use' must have shape \[3, 750\] or \[3, 2, 3, 125\], got \(3, 2, 125\)"):
        station_rf_samples(np.ones((S, 2, NT)), S, rf)
    one = _rf(gauss=[1.5])
    assert station_rf_samples(np.ones((S, 2, NT)), S, one).shape == (S, 2 * NT)
    assert station_rf_samples(np.ones((S, 2, 1, NT)), S, one).shape == (S, 2 * NT)
    for bad in (np.ones((S, 3, 2, NT)), np.ones((S, 2, 3, NT - 1)), np.ones((S, rf.nt + 1))):
        with pytest.raises(ValueError, match="'rf_use' must have shape"):
            station_rf_samples(bad, S, rf)
    with pytest.raises(ValueError, match="0/1"):
        station_rf_samples(np.full((S, 2, 3, NT), 2), S, rf)
    z = np.ones((S, 2, 3, NT))
    z[1] = 0
    with pytest.raises(ValueError, match="station 1 observes no receiver-function sample"):
        station_rf_samples(z, S, rf)


def test_rf_time_window_applies_a_rays_bounds_to_every_width():
    rf = _rf()
    u = rf_time_window(rf, np.array([[0.0, np.nan], [-5.0, 2.0], [1.0, 1.0]]), np.array([[10.0, 1.0], [40.0, 8.0],
                                                                                         [3.0, 3.0]]))
    assert u.shape == (S, rf.nt)
    u = u.reshape(S, 2, 3, NT)
    for g in range(3):
        assert np.array_equal(u[:, :, g], u[:, :, 0])
    one = rf_time_window(_rf(gauss=1.5), np.array([[0.0, np.nan], [-5.0, 2.0], [1.0, 1.0]]),
                         np.array([[10.0, 1.0], [40.0, 8.0], [3.0, 3.0]])).reshape(S, 2, NT)
    assert np.array_equal(u[:, :, 1], one) and not u[0, 1].any()


def test_loader_takes_the_width_shapes(tmp_path):
    rf = _rf()
    nd = _joint().ndata
    u = np.ones((S, 2, 3, NT), dtype=bool)
    u[2, 0] = False
    p = tmp_path / "st.npz"
    np.savez(p, dobs=np.zeros((S, nd)), rf_use=u)
    st = load_stations(str(p), nd, NP, driver_bounds(f1_true_model()), nray=2, rf=rf)
    assert np.array_equal(st["rf_use"], u.reshape(S, -1))
    st = load_stations({"dobs": np.zeros((S, nd)), "rf_use": u.reshape(S, -1)}, nd, NP,
                       driver_bounds(f1_true_model()), nray=2, rf=rf)
    assert np.array_equal(st["rf_use"], u.reshape(S, -1))
    with pytest.raises(ValueError, match="stations file: 'rf_use'.*shape"):
        load_stations({"dobs": np.zeros((S, nd)), "rf_use": u[:, :, 0]}, nd, NP, driver_bounds(f1_true_model()),
                      nray=2, rf=rf)


def test_station_models_need_a_product_of_rays_and_widths():
    u = np.ones((4, 2, 3, NT), dtype=bool)
    u[1, :, 1] = False            # width 2.5 missing on both rays: rays x {1.0, 5.0}
    u[2, 0] = False               # ray 0 missing: {0.06} x widths
    u[3, 0, 0] = False            # one (ray, width) trace missing: not a product
    sa = StationArray(_joint(), np.zeros((4, _joint().ndata)), rf_use=u)
    m = sa.station_model(1).rfmodel
    assert m.gauss == [1.0, 5.0] and m.ngauss == 2 and m.nray == 2 and m.nt == 4 * NT
    m = sa.station_model(2).rfmodel
    assert m.ray_p == 0.06 and m.gauss == WIDTHS and m.nt == 3 * NT
    assert sa.station_model(0).rfmodel.nt == 6 * NT
    with pytest.raises(ValueError, match=r"station 3 \(station0003\) observes different Gaussian widths.*station_view"):
        sa.station_model(3)
    w = u.copy()
    w[0, 1, 1, :5] = False       # a window: no station model, as with one width
    sw = StationArray(_joint(), np.zeros((4, _joint().ndata)), rf_use=w)
    with pytest.raises(ValueError, match="station 0 .* fits part of a receiver-function trace"):
        sw.station_model(0)
    # the station model's data are the observed traces in the array's order
    d = np.arange(_joint().ndata, dtype=np.float64)[None].repeat(4, axis=0)
    sd = StationArray(_joint(), d, rf_use=u)
    got = sd.station_model(1).dobs
    want = np.concatenate((d[1, :6 * NT].reshape(2, 3, NT)[:, [0, 2]].reshape(-1), d[1, 6 * NT:]))
    assert np.array_equal(got, want)
    # a scalar width stays a scalar in the one-width case
    one = StationArray(_joint(_rf(gauss=1.5)), np.zeros((2, 2 * NT + 72)), rf_use=np.ones((2, 2, NT), dtype=bool))
    assert one.station_model(0).rfmodel.gauss == 1.5
