"""Host side of the [vs, thk, vpvs] parameterisation (no GPU): argument checks, the driver's parameter-file
and stations-file paths up to the device call, the 3n initial-model rule of the samplers' restatement
(tests/vpvs_ref.py) and a finite-difference check of the composed reference objective's Vp/Vs gradient."""
import os
import numpy as np
import pytest
import yaml
from oracle import hmc_ref
import vpvs_ref
from oracle.oracle import brocher
from rfsurfhmc_b200.fixtures import (f1_config, f1_true_model, driver_bounds, driver_bounds_vpvs,
                                     sorted_uniform_models_vpvs)
from rfsurfhmc_b200.model.model_rf import ReceiverFunc
from rfsurfhmc_b200.model.model_surf import SurfWD
from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
from rfsurfhmc_b200.model.stations import StationArray
from rfsurfhmc_b200.pyhmc._common import station_run_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def x3_true():
    x = f1_true_model()
    vs = x[:7]
    vp, _ = brocher(vs)
    return np.hstack((x, vp / vs * 1.02))


def joint(vpvs=True):
    cfg = f1_config()
    rf = ReceiverFunc(cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], method="freq",
                      vpvs=vpvs)
    swd = SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"], vpvs=vpvs)
    return Joint_RF_SWD(1.0, 1.0, rf, swd)


def test_flag_defaults_off_and_init_reads_it():
    param = yaml.safe_load(open(os.path.join(G, "f1_param.yaml")))
    assert not ReceiverFunc.init(**param["rf"]).vpvs and not SurfWD.init(**param["swd"]).vpvs
    assert ReceiverFunc.init(**param["rf"], vpvs=True).npar == 3
    assert SurfWD.init(**param["swd"], vpvs=True).npar == 3
    m = joint()
    assert m.vpvs and m.npar == 3
    assert joint(False).npar == 2
    # the flag is part of the configuration key: flipping it reconfigures the device context
    a, b = joint(False), joint(True)
    assert a._config_fields(7) != b._config_fields(7)


def test_disagreeing_sub_models_are_rejected():
    cfg = f1_config()
    rf = ReceiverFunc(cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], vpvs=True)
    swd = SurfWD(tRc=cfg["tRc"], tRg=cfg["tRg"])
    with pytest.raises(ValueError, match="one parameterisation"):
        Joint_RF_SWD(1.0, 1.0, rf, swd)


@pytest.mark.parametrize("width", [14, 20, 22, 3])
def test_wrong_model_width_is_rejected_before_any_device_call(width):
    m = joint()
    with pytest.raises(ValueError, match="vpvs"):
        m.misfit_and_grad_batch(np.ones((2, width)))
    with pytest.raises(ValueError, match="vpvs"):
        m.rfmodel.misfit_and_grad_batch(np.ones((2, width)))
    with pytest.raises(ValueError, match="vpvs"):
        m.swdmodel.misfit_and_grad(np.ones(width))


def test_sampler_bounds_width_and_vpvs_box():
    m = joint()
    x = x3_true()
    b = driver_bounds_vpvs(x)
    assert b.shape == (21, 2)
    assert np.allclose(b[:14], driver_bounds(x[:14])) and np.allclose(b[14:, 0], 0.9 * x[14:])
    assert station_run_args(m, b, [0, 1], None) == (7, None)
    with pytest.raises(ValueError):
        station_run_args(m, driver_bounds(x[:14]), [0], None)       # [2n, 2] box for a 3n model
    bad = b.copy()
    bad[16, 0] = 1.0
    with pytest.raises(ValueError, match="lower bounds > 1"):
        station_run_args(m, bad, [0], None)
    # a station array: per-station boxes [S, 3n, 2], and station_model keeps the flag
    dobs = np.zeros((3, m.ndata))
    st = StationArray(m, dobs)
    assert st.vpvs and st.npar == 3
    assert station_run_args(st, np.stack([b] * 3), [0, 1], [0, 2])[0] == 7
    with pytest.raises(ValueError):
        st.misfit_and_grad_batch(np.ones((2, 14)), [0, 1])
    one = st.station_model(1)
    assert one.vpvs and one.rfmodel.vpvs and one.swdmodel.vpvs


def test_host_forward_uses_vp_from_vpvs(monkeypatch):
    """forward/misfit of the 3n vector: the drop-ins receive vp = k vs and Brocher rho of that vp."""
    from rfsurfhmc_b200.model import model_rf, model_surf
    seen = {}

    def rf_forward(thk, rho, vp, vs, *a):
        seen["rf"] = (thk, rho, vp, vs)
        return np.zeros(a[3])

    def surf_forward(thk, vp, vs, rho, *a):
        seen["swd"] = (thk, vp, vs, rho)
        return np.zeros(len(a[0])), True

    monkeypatch.setattr(model_rf.librf, "forward", rf_forward)
    monkeypatch.setattr(model_surf.libsurf, "forward", surf_forward)
    m = joint()
    x = x3_true()
    m.forward(x)
    vs, thk, k = x[:7], x[7:14], x[14:]
    vp = k * vs
    rho = 1.6612 * vp - 0.4721 * vp**2 + 0.0671 * vp**3 - 0.0043 * vp**4 + 0.000106 * vp**5
    for key, (t, r, a, b) in (("rf", seen["rf"]), ("swd", (seen["swd"][0], seen["swd"][3], seen["swd"][1],
                                                            seen["swd"][2]))):
        assert np.array_equal(t, thk) and np.array_equal(b, vs), key
        assert np.allclose(a, vp, rtol=1e-15) and np.allclose(r, rho, rtol=1e-14), key
    vp2, rho2, dadb, drda = m.swdmodel.empirical_relation(vs, deriv=True, k=k)
    assert np.allclose(vp2, vp) and np.allclose(dadb, k)


def _driver_param(tmp_path, vpvs):
    param = yaml.safe_load(open(os.path.join(G, "f1_param.yaml")))
    param["true_model"]["vpvs"] = list(vpvs)
    param["hmc"]["OUTPUT_DIR"] = str(tmp_path / "out")
    return param


class _Stop(Exception):
    pass


def _stub_device(monkeypatch):
    """The driver up to the sampler: no CUDA device, synthetic data captured, sampler init captured."""
    import torch
    from rfsurfhmc_b200 import driver
    seen = {}
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(driver.D, "bcast_array", lambda a, src=0: np.asarray(a))

    def fwd(self, x):
        seen["x"] = np.array(x)
        return np.zeros(self.rfmodel.nt), np.zeros(self.swdmodel.nt), True

    monkeypatch.setattr(Joint_RF_SWD, "forward", fwd)

    def init(cls, model, boundaries, rank, **kw):
        seen["model"], seen["bounds"] = model, np.array(boundaries)
        raise _Stop()

    monkeypatch.setattr(driver.HamitonianMC, "init", classmethod(init))
    return driver, seen


def test_driver_parameter_file_switches_to_vpvs(tmp_path, monkeypatch):
    driver, seen = _stub_device(monkeypatch)
    x = x3_true()
    with pytest.raises(_Stop):
        driver.run(_driver_param(tmp_path, x[14:]), nchains=2, save_chains=False)
    assert np.array_equal(seen["x"], x)            # observations synthesised from [vs, thk, vpvs]
    assert seen["model"].vpvs and seen["model"].npar == 3
    assert np.array_equal(seen["bounds"], driver_bounds_vpvs(x))
    with pytest.raises(ValueError, match="vpvs"):
        driver.run(_driver_param(tmp_path, x[14:20]), nchains=2, save_chains=False)


def test_driver_stations_file_takes_3n_boxes(tmp_path, monkeypatch):
    driver, seen = _stub_device(monkeypatch)
    x = x3_true()
    nd = 125 + 72
    b = np.stack([driver_bounds_vpvs(x), driver_bounds_vpvs(x * 1.01)])
    path = tmp_path / "st.npz"
    np.savez(path, dobs=np.zeros((2, nd)), bounds=b)
    with pytest.raises(_Stop):
        driver.run(_driver_param(tmp_path, x[14:]), nchains=2, save_chains=False, stations=str(path))
    assert isinstance(seen["model"], StationArray) and seen["model"].vpvs
    assert np.array_equal(seen["bounds"], b)
    np.savez(path, dobs=np.zeros((2, nd)), bounds=b[:, :14])
    with pytest.raises(ValueError, match="bounds"):
        driver.run(_driver_param(tmp_path, x[14:]), nchains=2, save_chains=False, stations=str(path))


def test_initial_model_rule_with_vpvs():
    x = x3_true()
    b = driver_bounds_vpvs(x)
    n = 7
    for seed in range(5):
        rs = np.random.RandomState(seed)
        x0 = vpvs_ref.initial_model(b, rs, npar=3)
        assert np.all(np.diff(x0[:n]) > 0)
        # redo the draws: the first box-valid draw, vs sorted and thk, vpvs permuted with it
        rs = np.random.RandomState(seed)
        while True:
            u = np.array([b[i, 0] + (b[i, 1] - b[i, 0]) * rs.rand() for i in range(3 * n)])
            idx = np.argsort(u[:n])
            y = np.concatenate([u[j * n:(j + 1) * n][idx] for j in range(3)])
            inside = (y >= b[:, 0]) & (y <= b[:, 1])
            inside[2 * n - 1] = True
            if inside.all():
                break
        assert np.array_equal(x0, y)
    # the default rule is unchanged: 2n boxes give what they always gave
    b2 = driver_bounds(x[:14])
    assert np.array_equal(hmc_ref._initial_model(b2, np.random.RandomState(3)),
                          vpvs_ref.initial_model(b2, np.random.RandomState(3), npar=2))
    X = sorted_uniform_models_vpvs(b, 16, seed=1)
    assert X.shape == (16, 21) and np.all(np.diff(X[:, :n], axis=1) > 0)


def test_composed_objective_gk_by_central_differences(oracle):
    cfg = f1_config()
    x = x3_true()
    dobs = vpvs_ref.vpvs_objective(oracle, x, np.zeros(125), cfg, which=1)[2]
    xp = x * (1 + 0.03 * np.sin(np.arange(21)))
    U, g, d, ok = vpvs_ref.vpvs_objective(oracle, xp, dobs, cfg, which=1)
    assert ok and g.shape == (21,) and U > 0
    h = 1e-6
    for j in (14, 16, 19):
        e = np.zeros(21)
        e[j] = h
        fd = (vpvs_ref.vpvs_objective(oracle, xp + e, dobs, cfg, which=1)[0] -
              vpvs_ref.vpvs_objective(oracle, xp - e, dobs, cfg, which=1)[0]) / (2 * h)
        assert abs(fd - g[j]) <= 1e-5 * np.max(np.abs(g[14:])), (j, fd, g[j])
    # with k = Brocher vp / vs the composition reproduces the oracle's own Brocher objective
    vs = xp[:7]
    xb = np.hstack((xp[:14], brocher(vs)[0] / vs))
    Ub, gb, db, _ = vpvs_ref.vpvs_objective(oracle, xb, dobs, cfg, which=1)
    U0, g0, d0, _ = oracle.joint_batch(xp[None, :14], dobs, cfg, which=1)
    assert np.isclose(Ub, U0[0], rtol=1e-10) and np.allclose(db, d0[0], rtol=1e-9, atol=1e-14)
    assert np.allclose(gb[7:14], g0[0, 7:], rtol=1e-8, atol=1e-12 * np.max(np.abs(g0)))
