"""Per-station SWD period lists, host side (no GPU): the stations-file key `swd_use` and the checks and
subset models StationArray makes before it touches a device."""
import numpy as np
import pytest
from rfsurfhmc_b200.fixtures import driver_bounds, f1_config, f1_true_model
from rfsurfhmc_b200.model.model_rf import ReceiverFunc
from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
from rfsurfhmc_b200.model.model_surf import SurfWD
from rfsurfhmc_b200.model.stations import StationArray, load_stations

S, NP = 3, 14
T = np.arange(5., 41.)


def _default():
    return driver_bounds(f1_true_model())


def _rf():
    cfg = f1_config()
    return ReceiverFunc(cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                        cfg["rf_type"], cfg["method"])


def _joint(swd=None):
    return Joint_RF_SWD(1.0, 1.0, _rf(), SurfWD(tRc=T, tRg=T.copy()) if swd is None else swd)


def _use(nper=72):
    u = np.ones((S, nper), dtype=bool)
    u[0, :5] = False        # no short Rc periods
    u[1, 36 + 30:] = False  # Rg ends early
    u[2, 36:] = False       # no Rg at all
    return u


def test_loader_accepts_per_station_periods(tmp_path):
    swd = SurfWD(tRc=T, tRg=T.copy())
    nd = _joint().ndata
    dobs = np.zeros((S, nd))
    assert load_stations({"dobs": dobs}, nd, NP, _default(), swd=swd)["swd_use"] is None
    path = tmp_path / "st.npz"
    np.savez(path, dobs=dobs, swd_use=_use().astype(np.int8))
    st = load_stations(str(path), nd, NP, _default(), swd=swd)
    assert st["swd_use"].dtype == bool and np.array_equal(st["swd_use"], _use())


@pytest.mark.parametrize("use,msg", [
    (np.ones((S, 71), dtype=bool), "shape"),        # wrong nper
    (np.ones((S - 1, 72), dtype=bool), "shape"),    # wrong station count
    (np.ones(72, dtype=bool), "shape"),
    (np.full((S, 72), 2), "0/1"),                    # not a mask
    (np.full((S, 72), 0.5), "0/1"),
    (np.vstack((np.ones((S - 1, 72)), np.zeros((1, 72)))), "observes no period"),
])
def test_loader_rejects_bad_masks_naming_the_key(use, msg):
    nd = _joint().ndata
    with pytest.raises(ValueError, match=f"stations file: 'swd_use'.*{msg}"):
        load_stations({"dobs": np.zeros((S, nd)), "swd_use": use}, nd, NP, _default(), swd=SurfWD(tRc=T, tRg=T))


def test_loader_needs_a_dispersion_configuration_for_the_mask():
    with pytest.raises(ValueError, match="'swd_use'"):
        load_stations({"dobs": np.zeros((S, 125)), "swd_use": np.ones((S, 72))}, 125, NP, _default())


def test_station_array_validates_masks_before_any_device():
    joint = _joint()
    dobs = np.zeros((S, joint.ndata))
    sa = StationArray(joint, dobs, swd_use=_use())
    assert sa.swd_use.dtype == bool and sa._ctx is None
    assert StationArray(joint, dobs).swd_use is None
    for bad in (_use()[:, 1:], _use()[1:], np.full((S, 72), 3)):
        with pytest.raises(ValueError, match="'swd_use'"):
            StationArray(joint, dobs, swd_use=bad)
    u = _use()
    u[1] = False
    with pytest.raises(ValueError, match="station 1 observes no period"):
        StationArray(joint, dobs, swd_use=u)
    rf = _rf()
    with pytest.raises(TypeError, match="swd_use"):
        StationArray(rf, np.zeros((S, rf.nt)), swd_use=_use())
    swd = SurfWD(tRc=T, tRg=T.copy())
    assert StationArray(swd, np.zeros((S, swd.nt)), swd_use=_use().astype(int)).swd_use.shape == (S, 72)


def test_love_mask_must_follow_the_rayleigh_phase_mask():
    """SurfWD evaluates Lc / Lg on tRc (model_surf.py _grad_periods): a station whose Love periods differ
    from its Rc periods has no single-station SurfWD."""
    t = T[:10]
    swd = SurfWD(tRc=t, tRg=t, tLc=t + 0.5, tLg=t + 0.25)
    d = np.zeros((S, swd.nt))
    u = np.ones((S, 40), dtype=bool)
    u[:, 0] = u[:, 20] = u[:, 30] = False  # the Rc, Lc and Lg masks agree; Rg may differ
    u[1, 10:13] = False
    assert StationArray(swd, d, swd_use=u).swd_use.shape == (S, 40)
    for col, w in ((25, "Lc"), (35, "Lg")):
        v = u.copy()
        v[2, col] = False
        with pytest.raises(ValueError, match=f"station 2 observes other {w} than Rc periods.*tRc"):
            StationArray(swd, d, swd_use=v)


def test_station_model_holds_the_subset_lists_and_compact_data():
    joint = _joint()
    nt = joint.rfmodel.nt
    dobs = np.arange(S * joint.ndata, dtype=np.float64).reshape(S, joint.ndata)
    sa = StationArray(joint, dobs, swd_use=_use())
    m = sa.station_model(0)
    assert np.array_equal(m.swdmodel.tRc, T[5:]) and m.swdmodel.ntRc == 31 and np.array_equal(m.swdmodel.tRg, T)
    assert m.swdmodel.nt == 67 and m.ndata == nt + 67
    assert np.array_equal(m.dobs, np.concatenate((dobs[0, :nt], dobs[0, nt + 5:])))
    m = sa.station_model(2)
    assert m.swdmodel.tRg is None and m.swdmodel.ntRg == 0 and m.ndata == nt + 36
    assert np.array_equal(m.dobs, dobs[2, :nt + 36])
    # the template keeps its grid
    assert joint.swdmodel.ntRc == 36 and joint.swdmodel.nt == 72
    # several modes: the mask applies to every mode block
    swd = SurfWD(mode=[0, 1], tRc=T, tRg=T.copy())
    d = np.arange(S * swd.nt, dtype=np.float64).reshape(S, swd.nt)
    m = StationArray(swd, d, swd_use=_use()).station_model(1)
    assert m.nt == 2 * 66
    assert np.array_equal(m.dobs, np.concatenate((d[1, :66], d[1, 72:138])))
