"""Per-station Gaussian widths, host side (no GPU): the stations-file key `gauss`, the checks
StationArray makes before it touches a device, and the widths station_model(s) carries."""
import numpy as np
import pytest
from rfsurfhmc_b200.fixtures import driver_bounds, f1_config, f1_true_model
from rfsurfhmc_b200.model.model_rf import ReceiverFunc
from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
from rfsurfhmc_b200.model.model_surf import SurfWD
from rfsurfhmc_b200.model.stations import StationArray, load_stations, station_gauss

ND, NP, S = 197, 14, 3


def _default():
    return driver_bounds(f1_true_model())


def _rf(gauss, rays=0.045):
    cfg = f1_config()
    return ReceiverFunc(rays, cfg["nt"], cfg["dt"], gauss, cfg["time_shift"], cfg["water"], cfg["rf_type"],
                        cfg["method"])


def _joint(gauss, rays=0.045):
    cfg = f1_config()
    return Joint_RF_SWD(1.0, 1.0, _rf(gauss, rays), SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"]))


def test_loader_accepts_per_station_widths(tmp_path):
    dobs = np.zeros((S, ND))
    st = load_stations({"dobs": dobs}, ND, NP, _default())
    assert st["gauss"] is None
    g = np.array([1.0, 2.5, 1.5])
    st = load_stations({"dobs": dobs, "gauss": g}, ND, NP, _default())
    assert st["gauss"].shape == (S, 1) and st["gauss"].dtype == np.float64 and np.array_equal(st["gauss"][:, 0], g)
    assert np.array_equal(load_stations({"dobs": dobs, "gauss": g[:, None]}, ND, NP, _default())["gauss"],
                          st["gauss"])
    g2 = np.array([[1.0, 2.5], [1.5, 3.0], [2.0, 5.0]])
    assert np.array_equal(load_stations({"dobs": dobs, "gauss": g2}, ND, NP, _default(), ngauss=2)["gauss"], g2)
    path = tmp_path / "st.npz"
    np.savez(path, dobs=dobs, gauss=g2)
    assert np.array_equal(load_stations(str(path), ND, NP, _default(), ngauss=2)["gauss"], g2)
    np.savez(path, dobs=dobs, gauss=g)
    assert np.array_equal(load_stations(str(path), ND, NP, _default())["gauss"][:, 0], g)


@pytest.mark.parametrize("gauss,ngauss", [
    (np.full(2, 1.5), 1),                # wrong station count
    (np.full(4, 1.5), 1),
    (np.full((S, 2), 1.5), 1),           # two widths for a one-width objective
    (np.full(S, 1.5), 2),                # one width for a two-width objective
    (np.full((S, 3), 1.5), 2),
    (np.full((S, 2, 1), 1.5), 2),        # extra dimension
    (np.full((S, 1, 1), 1.5), 1),
    (np.float64(1.5), 1),                # a scalar
    (np.array([1.5, 0.0, 2.5]), 1),      # not positive
    (np.array([1.5, -1.0, 2.5]), 1),
    (np.array([1.5, np.nan, 2.5]), 1),
    (np.array([[1.0, 2.5], [np.inf, 2.5], [1.0, 2.5]]), 2),
    (np.array([[1.0, 2.5], [1.0, -np.inf], [1.0, 2.5]]), 2),
])
def test_loader_rejects_bad_widths_naming_the_key(gauss, ngauss):
    with pytest.raises(ValueError, match="stations file: 'gauss'"):
        load_stations({"dobs": np.zeros((S, ND)), "gauss": gauss}, ND, NP, _default(), ngauss=ngauss)
    with pytest.raises(ValueError, match="^'gauss'"):
        station_gauss(gauss, S, ngauss)


def test_station_array_validates_widths_before_any_device():
    joint = _joint(1.5)
    dobs = np.zeros((S, joint.ndata))
    sa = StationArray(joint, dobs, gauss=[1.0, 2.5, 1.5])
    assert sa.gauss.shape == (S, 1) and sa._ctx is None
    assert StationArray(joint, dobs).gauss is None
    for bad in ([1.0, 2.5], [1.0, 0.0, 2.5], [1.0, np.nan, 2.5], np.full((S, 2), 1.5)):
        with pytest.raises(ValueError, match="'gauss'"):
            StationArray(joint, dobs, gauss=bad)
    two = _joint([1.0, 2.5])
    d2 = np.zeros((S, two.ndata))
    assert StationArray(two, d2, gauss=np.full((S, 2), 2.0)).gauss.shape == (S, 2)
    with pytest.raises(ValueError, match="'gauss'"):
        StationArray(two, d2, gauss=np.full(S, 2.0))
    rf = _rf([1.0, 2.5])
    assert StationArray(rf, np.zeros((S, rf.nt)), gauss=np.full((S, 2), 2.0)).gauss.shape == (S, 2)
    cfg = f1_config()
    swd = SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"])
    with pytest.raises(TypeError, match="gauss"):
        StationArray(swd, np.zeros((S, swd.nt)), gauss=np.full(S, 2.0))


def test_station_model_carries_each_stations_widths():
    # a scalar template width gives a scalar, a list gives a list; the template is left as it was
    joint = _joint(1.5)
    g1 = np.array([1.0, 2.5, 2.0])
    sa = StationArray(joint, np.arange(S * joint.ndata, dtype=np.float64).reshape(S, -1), gauss=g1)
    for s in range(S):
        m = sa.station_model(s)
        assert m.rfmodel.gauss == g1[s] and isinstance(m.rfmodel.gauss, float)
        assert m.rfmodel.ngauss == 1 and m.rfmodel.ray_p == joint.rfmodel.ray_p
        assert np.array_equal(m.rfobs, sa.dobs[s, :joint.rfmodel.nt])
    assert joint.rfmodel.gauss == 1.5
    rf = _rf([1.0, 2.5])
    g2 = np.array([[1.0, 2.5], [1.5, 3.0], [0.5, 2.0]])
    sa = StationArray(rf, np.zeros((S, rf.nt)), gauss=g2)
    for s in range(S):
        m = sa.station_model(s)
        assert m.gauss == g2[s].tolist() and m.ngauss == 2 and m.nt == rf.nt
    assert rf.gauss == [1.0, 2.5]
    one = _rf([2.0])  # a one-width list stays a list
    sa = StationArray(one, np.zeros((S, one.nt)), gauss=g1)
    assert sa.station_model(1).gauss == [2.5]


def test_station_model_with_rf_use_keeps_the_stations_remaining_widths():
    rf = _rf([1.0, 2.5], rays=[0.04, 0.06])
    nt = rf.nt_trace
    g2 = np.array([[1.0, 2.5], [1.5, 3.0], [0.5, 2.0]])
    use = np.ones((S, 2, 2, nt), dtype=bool)
    use[1, :, 0] = False  # station 1 fits its second width only
    use[2, :, 1] = False  # station 2 its first
    dobs = np.arange(S * rf.nt, dtype=np.float64).reshape(S, -1)
    sa = StationArray(rf, dobs, rf_use=use, gauss=g2)
    assert sa.station_model(0).gauss == [1.0, 2.5]
    m1, m2 = sa.station_model(1), sa.station_model(2)
    assert m1.gauss == [3.0] and m1.ngauss == 1 and m1.nt == 2 * nt
    assert m2.gauss == [0.5] and m2.ngauss == 1
    assert np.array_equal(m1.dobs, dobs[1].reshape(2, 2, nt)[:, 1].reshape(-1))
    assert rf.gauss == [1.0, 2.5] and rf.ngauss == 2
