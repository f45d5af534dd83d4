"""Per-station ray parameters, host side (no GPU): the stations-file key `ray_p` and the checks
StationArray makes before it touches a device."""
import numpy as np
import pytest
from rfsurfhmc_b200.fixtures import driver_bounds, f1_config, f1_true_model
from rfsurfhmc_b200.model.model_rf import ReceiverFunc
from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
from rfsurfhmc_b200.model.model_surf import SurfWD
from rfsurfhmc_b200.model.stations import StationArray, load_stations

ND, NP, S = 197, 14, 3


def _default():
    return driver_bounds(f1_true_model())


def _rf(rays):
    cfg = f1_config()
    return ReceiverFunc(rays, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                        cfg["rf_type"], cfg["method"])


def _joint(rays):
    cfg = f1_config()
    return Joint_RF_SWD(1.0, 1.0, _rf(rays), SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"]))


def test_loader_accepts_per_station_rays(tmp_path):
    dobs = np.zeros((S, ND))
    st = load_stations({"dobs": dobs}, ND, NP, _default())
    assert st["ray_p"] is None
    p = np.array([0.045, 0.06, 0.07])
    st = load_stations({"dobs": dobs, "ray_p": p}, ND, NP, _default())
    assert st["ray_p"].shape == (S, 1) and np.array_equal(st["ray_p"][:, 0], p)
    assert np.array_equal(load_stations({"dobs": dobs, "ray_p": p[:, None]}, ND, NP, _default())["ray_p"],
                          st["ray_p"])
    p2 = np.array([[0.04, 0.06], [0.05, 0.07], [0.045, 0.065]])
    path = tmp_path / "st.npz"
    np.savez(path, dobs=dobs, ray_p=p2)
    st = load_stations(str(path), ND, NP, _default(), nray=2)
    assert np.array_equal(st["ray_p"], p2)


@pytest.mark.parametrize("ray_p,nray", [
    (np.full(2, 0.06), 1),             # wrong station count
    (np.full((S, 2), 0.06), 1),        # two rays for a one-ray objective
    (np.full(S, 0.06), 2),             # one ray for a two-ray objective
    (np.full((S, 3), 0.06), 2),
    (np.full((S, 2, 1), 0.06), 2),
    (np.float64(0.06), 1),
    (np.array([0.06, 0.0, 0.07]), 1),  # not positive
    (np.array([0.06, -0.05, 0.07]), 1),
    (np.array([0.06, np.nan, 0.07]), 1),
    (np.array([[0.06, 0.05], [np.inf, 0.06], [0.07, 0.07]]), 2),
])
def test_loader_rejects_bad_rays_naming_the_key(ray_p, nray):
    with pytest.raises(ValueError, match="stations file: 'ray_p'"):
        load_stations({"dobs": np.zeros((S, ND)), "ray_p": ray_p}, ND, NP, _default(), nray=nray)


def test_station_array_validates_rays_before_any_device():
    cfg = f1_config()
    joint = _joint(cfg["ray_p"])
    dobs = np.zeros((S, joint.ndata))
    sa = StationArray(joint, dobs, ray_p=[0.05, 0.06, 0.07])
    assert sa.ray_p.shape == (S, 1) and sa._ctx is None
    assert StationArray(joint, dobs).ray_p is None
    with pytest.raises(ValueError, match="'ray_p'"):
        StationArray(joint, dobs, ray_p=[0.05, 0.06])
    with pytest.raises(ValueError, match="'ray_p'"):
        StationArray(joint, dobs, ray_p=[0.05, 0.0, 0.07])
    two = _joint([0.04, 0.06])
    d2 = np.zeros((S, two.ndata))
    assert StationArray(two, d2, ray_p=np.full((S, 2), 0.05)).ray_p.shape == (S, 2)
    with pytest.raises(ValueError, match="'ray_p'"):
        StationArray(two, d2, ray_p=np.full(S, 0.05))
    rf = _rf(cfg["ray_p"])
    assert StationArray(rf, np.zeros((S, rf.nt)), ray_p=np.full(S, 0.05)).ray_p.shape == (S, 1)
    swd = SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"])
    with pytest.raises(TypeError, match="ray_p"):
        StationArray(swd, np.zeros((S, swd.nt)), ray_p=np.full(S, 0.05))


def test_station_model_carries_its_own_rays():
    cfg = f1_config()
    sa = StationArray(_joint(cfg["ray_p"]), np.zeros((S, _joint(cfg["ray_p"]).ndata)), ray_p=[0.05, 0.06, 0.07])
    m = sa.station_model(1)
    assert m.rfmodel.ray_p == 0.06 and isinstance(m.rfmodel.ray_p, float)
    assert sa.template.rfmodel.ray_p == cfg["ray_p"]
    two = _joint([0.04, 0.06])
    p2 = np.array([[0.041, 0.061], [0.042, 0.062], [0.043, 0.063]])
    m = StationArray(two, np.zeros((S, two.ndata)), ray_p=p2).station_model(2)
    assert m.rfmodel.ray_p == [0.043, 0.063] and two.rfmodel.ray_p == [0.04, 0.06]
    rf = _rf(cfg["ray_p"])
    assert StationArray(rf, np.zeros((S, rf.nt)), ray_p=[0.05, 0.06, 0.07]).station_model(2).ray_p == 0.07
    # without a table, the copies keep the template's value
    assert StationArray(rf, np.zeros((S, rf.nt))).station_model(0).ray_p == cfg["ray_p"]
