"""Oracle vs committed golden vectors, the C ABI surface, host-side logic (no GPU needed)."""
import ctypes
import os
import re
import numpy as np
import pytest
from oracle.oracle import brocher
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, sorted_uniform_models

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def test_oracle_reproduces_dropin_golden(oracle):
    g = np.load(os.path.join(G, "f1_dropin.npz"))
    thk, vs, vp, rho, T = g["thk"], g["vs"], g["vp"], g["rho"], g["T"]
    for wt in ("Rc", "Rg", "Lc", "Lg"):
        for mode in (0, 1, 2):
            c, ok = oracle.surf_forward(thk, vp, vs, rho, T, wt, mode=mode)
            assert ok == bool(g[f"fwd_{wt}_{mode}_ok"])
            assert np.allclose(c, g[f"fwd_{wt}_{mode}"], rtol=1e-12, atol=0, equal_nan=True)
        r = oracle.surf_adjoint_kernel(thk, vp, vs, rho, T, wt)
        for arr, key in zip(r[:5], ("c", "da", "db", "dr", "dh")):
            assert np.allclose(arr, g[f"ker_{wt}_{key}"], rtol=1e-10, atol=1e-14)
    q = thk * 0 + 9999.
    for rft in ("P", "S"):
        rf, kl = oracle.rf_kernel_all(thk, rho, vp, vs, q, q, 0.045, 125, 0.4, 1.5, 5.0, "freq", 0.001, rft)
        assert np.allclose(rf, g[f"rf_{rft}"], rtol=1e-10, atol=1e-13)
        assert np.allclose(kl, g[f"rf_{rft}_kl"], rtol=1e-9, atol=1e-12)


def test_oracle_reproduces_joint_golden(oracle):
    g = np.load(os.path.join(G, "f1_joint.npz"))
    U, gr, d, f = oracle.joint_batch(g["X"][:16], g["dobs"], f1_config(), nthreads=4)
    assert np.array_equal(f, g["flag"][:16])
    assert np.allclose(U, g["U"][:16], rtol=1e-10)
    assert np.allclose(gr, g["grad"][:16], rtol=1e-8, atol=1e-10)


def test_joint_glue_matches_numpy_restatement(oracle):
    """Joint_RF_SWD.misfit_and_grad assembled in NumPy from the drop-in calls
    (model_rf.py:182-193, model_surf.py:175-224, model_rf_swd_vs_thk.py:66-86) == oracle batch glue."""
    cfg = f1_config()
    x0 = f1_true_model()
    _, _, dd, _ = oracle.joint_batch(x0[None, :], np.zeros(197), cfg)
    dobs = dd[0]
    x = sorted_uniform_models(driver_bounds(x0), 1, seed=5)[0]
    vs, thk = x[:7], x[7:]
    vp, rho = brocher(vs)
    drda = 1.6612 - 0.4721 * 2 * vp + 0.0671 * 3 * vp**2 - 0.0043 * 4 * vp**3 + 0.000106 * 5 * vp**4
    dadb = 2.0947 - 0.8206 * 2 * vs + 0.2683 * 3 * vs**2 - 0.0251 * 4 * vs**3
    q = thk * 0 + 9999.
    d, kl = oracle.rf_kernel_all(thk, rho, vp, vs, q, q, 0.045, 125, 0.4, 1.5, 5.0, "freq", 0.001, "P")
    K = kl[2] + dadb[:, None] * kl[1] + (drda * dadb)[:, None] * kl[0]
    r = d - dobs[:125]
    g_rf = np.hstack((K @ r, kl[3] @ r))
    U_rf = 0.5 * np.sum(r**2)
    ds = np.zeros(72); Kv = np.zeros((72, 7)); Kh = np.zeros((72, 7))
    for i, wt in enumerate(("Rc", "Rg")):
        c, da, db, dr, dh, ok = oracle.surf_adjoint_kernel(thk, vp, vs, rho, cfg["tRc"], wt)
        assert ok
        ds[36 * i:36 * i + 36] = c
        Kv[36 * i:36 * i + 36] = db + da * dadb + dr * drda * dadb
        Kh[36 * i:36 * i + 36] = dh
    rs = ds - dobs[125:]
    g_sw = np.hstack((rs @ Kv, rs @ Kh))
    wt = 125 / 72
    U, g, dsyn, f = oracle.joint_batch(x[None, :], dobs, cfg)
    assert f[0]
    assert np.isclose(U[0], U_rf + wt * 0.5 * np.sum(rs**2), rtol=1e-12)
    assert np.allclose(g[0], g_rf + wt * g_sw, rtol=1e-10, atol=1e-12)
    assert np.allclose(dsyn[0], np.hstack((d, ds)), rtol=1e-13)


def test_cabi_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "rfsurfhmc.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(rfs_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 18
    from rfsurfhmc_b200 import _lib
    assert set(_lib.exported_symbols()) == declared
    lib = ctypes.CDLL(_lib.LIB_PATH)  # loads without a GPU (no compute calls here)
    for s in declared:
        assert hasattr(lib, s), s
    lib.rfs_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.rfs_version()


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from rfsurfhmc_b200._lib import Context, RfsError
    with pytest.raises(RfsError):
        Context(0)
    from rfsurfhmc_b200.model.lib import libsurf
    with pytest.raises(RfsError):
        libsurf.forward([1., 0.], [5., 6.], [3., 3.5], [2.5, 2.8], [5.], "Rc")
    with pytest.raises(ValueError):
        libsurf.forward([1., 0.], [5., 6.], [3., 3.5], [2.5, 2.8], [5.], "Zz")


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rfsurfhmc_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".inl", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("no oracle", ""), os.path.join(dp, f)


def test_driver_bounds_and_initial_model_distribution():
    x0 = f1_true_model()
    b = driver_bounds(x0)
    assert b.shape == (14, 2)
    assert np.all(b[:7, 0] >= 1.5) and np.all(b[:7, 1] <= 5.0)
    assert tuple(b[-1]) == (0.0, 2.0)
    assert np.allclose(b[7:13, 0], x0[7:13] * 0.8) and np.allclose(b[7:13, 1], x0[7:13] * 1.2)
    X = sorted_uniform_models(b, 100, 0)
    assert np.all(np.diff(X[:, :7], axis=1) >= 0)


def test_hmc_reference_restatement_on_quadratic_model():
    """hmc_ref (the checker of the device sampler) samples a Gaussian correctly and its random
    stream is NumPy's legacy one (first draws equal np.random after the same seed)."""
    from oracle import hmc_ref
    n2 = 4
    bounds = np.tile(np.array([[-5., 5.]]), (n2, 1))
    f = lambda x: (0.5 * float(x @ x), x.copy(), np.zeros(3), True)
    R = hmc_ref.run_base(f, bounds, 0.3, (5, 20), 42, nsamples=400, ndraws=100)
    assert R.n_acc == 500 and len(R.accepts) == R.n_iter
    # reference quirk Q9: momenta are drawn with variance 0.25 but K = p.p/2 (unit mass), so the
    # chain equilibrates at an effective temperature of 0.25 -> sample variance ~0.25, not 1
    assert 0.15 < np.var(R.samples) < 0.40
    # the random stream is NumPy's legacy global one: the initial model is built from the first
    # n2 np.random.rand() draws after np.random.seed(seed)
    np.random.seed(42)
    u = np.array([np.random.rand() for _ in range(n2)])
    x = bounds[:, 0] + 10 * u
    idx = np.argsort(x[:2])
    expect = np.hstack((x[:2][idx], x[2:][idx]))
    assert np.allclose(R.initmodel, expect)
    R2 = hmc_ref.run_da(f, bounds, 0.1, 10, 0.65, 43, nsamples=300, ndraws=100)
    assert R2.n_acc == 400
    assert 0.4 < np.mean(R2.accepts[150:]) < 0.9


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` runs the CPU restatement on the host cores (no GPU needed) and
    prints ONE JSON line with the keys the driver reads."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "3"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "evals/s" and line["value"] > 0
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "evals/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_bench_dump_outputs_writes_floats_and_a_fixed_sample_above_the_cap(tmp_path):
    """`bench.py --dump-outputs DIR`: one .npy per output in float64 (flag in float32); above the size
    cap every array keeps the same seeded sample of chains, listed in rows.npy, from run to run."""
    import torch
    import bench
    B = 1000
    t = {"U": torch.arange(B, dtype=torch.float64), "grad": torch.arange(B * 14, dtype=torch.float64).reshape(B, 14),
         "flag": torch.ones(B, dtype=torch.uint8)}
    bench.dump_outputs(str(tmp_path / "all"), t)
    assert sorted(os.listdir(tmp_path / "all")) == ["U.npy", "flag.npy", "grad.npy"]
    full = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in t}
    assert full["U"].dtype == np.float64 and full["grad"].dtype == np.float64 and full["flag"].dtype == np.float32
    assert np.array_equal(full["grad"], t["grad"].numpy()) and np.all(full["flag"] == 1)
    cap = 50000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), t, limit=cap)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= cap
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and 100 < len(rows) < B and np.all(np.diff(rows) > 0)
    for k in ("U", "grad", "flag", "rows"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy"))
    r = rows.astype(int)
    assert np.array_equal(np.load(tmp_path / "a" / "U.npy"), full["U"][r])
    assert np.array_equal(np.load(tmp_path / "a" / "grad.npy"), full["grad"][r])


def test_chain_result_file_and_best_mean_model(tmp_path):
    """Per-chain result file (logical HDF5 layout of pyhmc/hmc.py:203-226 in an .npz) and the
    nbest-average model (hmc.py:266-270); samplers refuse models without a device context."""
    from rfsurfhmc_b200.pyhmc._common import write_chain_file, best_mean_model, require_device_model
    rng = np.random.default_rng(3)
    samples, syn = rng.random((12, 6)), rng.random((12, 9))
    misfit = rng.random(12)
    xm = best_mean_model(misfit, samples, 4)
    assert np.allclose(xm, samples[np.argsort(misfit)[:4]].mean(axis=0))
    path = tmp_path / "sub" / "chain_x.0.npz"
    write_chain_file(str(path), samples[0], syn[0], xm, syn.mean(0), samples, syn)
    z = np.load(path)
    assert sorted(z.files) == sorted(["initmodel", "obs", "mean/model", "mean/syn", "models", "syn", "complete"])
    assert np.array_equal(z["models"], samples) and np.array_equal(z["mean/model"], xm) and bool(z["complete"])
    with pytest.raises(TypeError):
        require_device_model(object())


def test_incomplete_chains_are_masked_and_flagged(tmp_path):
    """A chain stopped by max_iters (or stuck at a failing state) leaves rows unfilled: they must not
    look like zero-misfit samples (the 'best' ones for argsort), the accept ratio must count what was
    run, and the chain file must say it is incomplete (ADVICE r1, driver.py)."""
    import warnings
    from rfsurfhmc_b200.pyhmc._common import finish_run, save_chain, best_mean_model
    ns, nd, n2 = 5, 2, 4
    out = {"misfit": np.array([[3., 2., 0., 0., 0.], [5., 4., 3., 2., 1.]]),
           "samples": np.arange(2 * ns * n2, dtype=float).reshape(2, ns, n2), "syn": None,
           "initmodel": np.zeros((2, n2)), "n_acc": np.array([4, 7]), "n_iter": np.array([9, 8]),
           "warning": "1 chain(s) stuck"}
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        finish_run(out, ns, nd)
    assert len(w) == 2 and "stuck" in str(w[0].message)
    assert out["n_valid"].tolist() == [2, 5] and out["complete"].tolist() == [False, True]
    assert np.isnan(out["misfit"][0, 2:]).all() and np.isfinite(out["misfit"][1]).all()
    xm = best_mean_model(out["misfit"][0], out["samples"][0], 3, out["n_valid"][0])
    assert np.allclose(xm, out["samples"][0][:2].mean(axis=0))      # the zero rows are not 'best'

    class M:
        dobs = np.zeros(3)

        def misfit_and_grad(self, x):
            return 0.0, x, np.ones(3)
    save_chain(str(tmp_path / "c.0.npz"), M(), out, 0, 3, ns)
    z = np.load(tmp_path / "c.0.npz")
    assert not bool(z["complete"]) and z["models"].shape == (2, n2)


def _ref_python_golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_code.npz"))


def test_restated_cpp_layers_match_the_references_own_compiled_modules(oracle):
    """The fixture holds the outputs of the reference's OWN pybind11 modules -- src/SWD/main.cpp +
    surfdisp.cpp and src/RF/main.cpp compiled in place (`make -C oracle ref`), their Fortran entry
    points forwarded to the restated routines.  The oracle's restatement of those C++ layers
    (swd_driver.cpp, oracle_capi.cpp: float32 casts, retry loop, group-velocity drivers, kernel
    driver, flat->sphere conversion, argument conventions) must agree bit for bit."""
    z = _ref_python_golden()
    T = z["cpp_T"]
    n = 0
    for im, (h, a, v, r) in enumerate(z["cpp_models"]):
        for wt in ("Rc", "Rg", "Lc", "Lg"):
            for mode in (0, 1, 2):
                for sph in (False, True):
                    key = f"cpp{im}_{wt}_{mode}_{int(sph)}"
                    if key + "_fwd" not in z.files:
                        continue
                    c, ok = oracle.surf_forward(h, a, v, r, T, wt, mode, sph)
                    k = oracle.surf_adjoint_kernel(h, a, v, r, T, wt, mode, sph)
                    assert [ok, k[5]] == z[key + "_ok"].tolist(), key
                    assert np.array_equal(c, z[key + "_fwd"], equal_nan=True), key
                    for nm, arr in zip(("c", "da", "db", "dr", "dh"), k[:5]):
                        if key + "_k" + nm in z.files:
                            assert np.array_equal(arr, z[key + "_k" + nm], equal_nan=True), (key, nm)
                    n += 1
    assert n == 24 + 3 * 8
    thk, vp, vs, rho = z["cpp_models"][0]
    q = thk * 0 + 9999.0
    rfa = (0.045, 125, 0.4, 1.5, 5.0)
    for method in ("freq", "time"):
        for rft in ("P", "S"):
            key = f"cpprf_{method}_{rft}"
            assert np.array_equal(oracle.rf_forward(thk, rho, vp, vs, q, q, *rfa, method, 0.001, rft), z[key + "_fwd"])
            assert np.array_equal(oracle.rf_kernel_all(thk, rho, vp, vs, q, q, *rfa, method, 0.001, rft)[1], z[key + "_all"])
            for par in ("vs", "vp", "rho", "thick"):
                assert np.array_equal(oracle.rf_kernel(thk, rho, vp, vs, q, q, *rfa, method, 0.001, rft, par)[1],
                                      z[key + "_k" + par])


def test_restated_glue_matches_the_references_own_python(oracle):
    """tests/golden/reference_code.npz was produced by the reference's UNMODIFIED model/*.py classes
    (imported from /root/reference by tests/golden/make_reference_golden.py) on top of oracle-backed
    libsurf/librf stubs.  The restated glue of the oracle (Brocher relations, chain rule, residual
    contraction, 125/72 joint weighting, failure convention) must give the same numbers."""
    z = _ref_python_golden()
    cfg = f1_config()
    X, dobs = z["glue_X"], z["dobs"]
    U, g, d, f = oracle.joint_batch(X, dobs, cfg, which=0)
    assert np.array_equal(f, z["glue_flag"])
    assert np.allclose(U, z["glue_U"], rtol=1e-12, atol=0)
    assert np.allclose(g, z["glue_grad"], rtol=1e-10, atol=1e-12 * np.abs(z["glue_grad"]).max())
    assert np.allclose(d, z["glue_dsyn"], rtol=1e-13, atol=1e-15)
    Ur, gr, _, _ = oracle.joint_batch(X, dobs[:125], cfg, which=1)
    Us, gs, _, _ = oracle.joint_batch(X, dobs[125:], cfg, which=2)
    assert np.allclose(Ur, z["glue_U_rf"], rtol=1e-12) and np.allclose(Us, z["glue_U_swd"], rtol=1e-12)
    assert np.allclose(gr, z["glue_grad_rf"], rtol=1e-10, atol=1e-12 * np.abs(z["glue_grad_rf"]).max())
    assert np.allclose(gs, z["glue_grad_swd"], rtol=1e-10, atol=1e-12 * np.abs(z["glue_grad_swd"]).max())


def test_restated_samplers_match_the_references_own_python(oracle):
    """Same fixture: HamitonianMC.sample / HMCDualAveraging.sample of the reference ran on the joint
    model; oracle/hmc_ref.py (the checker of the device sampler) must reproduce the initial model,
    every L, every step size, every acceptance probability / decision and every returned state."""
    from oracle import hmc_ref
    z = _ref_python_golden()
    cfg = f1_config()
    f = hmc_ref.oracle_joint_f(oracle, z["dobs"], cfg)
    b = z["bounds"]
    assert np.array_equal(b, driver_bounds(z["x_true"]))
    dt, l0, l1, seed, ns, ndr = z["base_hparam"]
    for rank in (0, 3):
        acc = z[f"base{rank}_accepts"]
        R = hmc_ref.run_base(f, b, float(dt), (int(l0), int(l1)), int(seed) + rank, nsamples=int(ns),
                             ndraws=int(ndr), max_iters=len(acc))
        assert np.array_equal(R.initmodel, z[f"base{rank}_init"])
        assert R.accepts == acc.tolist() and R.trace_L == z[f"base{rank}_L"].tolist()
        assert np.allclose(np.array(R.trace_x), z[f"base{rank}_x"], rtol=1e-12, atol=1e-13)
    dt, L0, target, seed, ns, ndr = z["da_hparam"]
    for rank in (0, 5):
        Ls = z[f"da{rank}_L"]
        R = hmc_ref.run_da(f, b, float(dt), int(L0), float(target), int(seed) + rank, nsamples=int(ns),
                           ndraws=int(ndr), max_iters=len(Ls))
        assert np.array_equal(R.initmodel, z[f"da{rank}_init"])
        assert R.trace_L == Ls.tolist()
        assert np.allclose(R.trace_dt, z[f"da{rank}_dt"], rtol=1e-12)
        assert np.allclose(R.trace_alpha, z[f"da{rank}_alpha"], rtol=1e-9, atol=1e-300)
        assert np.allclose(np.array(R.trace_x), z[f"da{rank}_x"], rtol=1e-12, atol=1e-13)


def test_reference_drivers_end_to_end_match_the_restatement(oracle):
    """main_base.py and main_DA.py of the reference ran UNMODIFIED as __main__ (one MPI rank, short
    chains) for the fixture: the bounds they build, the observations they synthesise (real_syn.npy)
    and the misfit history they save (misfit.npy) must come out of driver_bounds, the oracle's
    forward and hmc_ref."""
    from oracle import hmc_ref
    z = _ref_python_golden()
    cfg = f1_config()
    x0 = f1_true_model()
    for tag in ("drvbase", "drvda"):
        assert np.array_equal(z[tag + "_bounds"], driver_bounds(x0))
        _, _, d0, f0 = oracle.joint_batch(x0[None, :], np.zeros(197), cfg, which=0)
        assert f0[0] and np.allclose(d0[0], z[tag + "_real_syn"], rtol=1e-13, atol=1e-15)
    f = hmc_ref.oracle_joint_f(oracle, z["drvbase_real_syn"], cfg)
    ns, ndr, dt = z["drvbase_cfg"]
    R = hmc_ref.run_base(f, driver_bounds(x0), float(dt), (5, 20), 991206, nsamples=int(ns), ndraws=int(ndr))
    assert R.n_acc == int(ns + ndr)
    assert np.allclose(R.misfit, z["drvbase_misfit"][0], rtol=1e-9)
    ns, ndr, dt = z["drvda_cfg"]
    R = hmc_ref.run_da(f, driver_bounds(x0), float(dt), 10, 0.65, 991206, nsamples=int(ns), ndraws=int(ndr))
    assert R.n_acc == int(ns + ndr)
    assert np.allclose(R.misfit, z["drvda_misfit"][0], rtol=1e-9)


def test_references_own_test_script_curves(oracle):
    """test_forward.py -- the only test the reference ships -- ran unmodified for the fixture
    (time-domain RF with nt=500, dt=0.1, a=1.0; Rc and Rg at 5..40 s for its second model).  The
    oracle's Python API must give the curves it plots."""
    z = _ref_python_golden()
    thk = np.array([6., 6, 13, 5, 10, 30, 0]); vs = np.array([3.2, 3.4, 3.46, 3.7, 3.9, 4.5, 4.7])
    vp, rho = brocher(vs)
    q = thk * 0 + 9999.
    rf = oracle.rf_forward(thk, rho, vp, vs, q, q, 0.045, 500, 0.1, 1.0, 5.0, "time", 0.001, "P")
    assert np.array_equal(rf, z["tf_rf"]) and np.allclose(z["tf_t"], np.arange(500) * 0.1 - 5.0)
    T = z["tf_tRc"]
    assert np.array_equal(oracle.surf_forward(thk, vp, vs, rho, T, "Rc")[0], z["tf_Rc"])
    assert np.array_equal(oracle.surf_forward(thk, vp, vs, rho, T, "Rg")[0], z["tf_Rg"])


def test_real_data_resampling_matches_the_references_own_utils():
    """rfsurfhmc_b200/utils.py against outputs of the reference's unmodified src/utils.py
    (tests/golden/make_utils_golden.py generated utils_resample.npz in the build container)."""
    from rfsurfhmc_b200.utils import get_rf_inv_para, next_power_of_2
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "utils_resample.npz"))
    assert [next_power_of_2(int(v)) for v in z["pow2_in"]] == z["pow2_out"].tolist()
    for i in range(3):
        ts, te = z[f"in_{i}_win"]
        y, nt, dt, shift = get_rf_inv_para(z[f"in_{i}_d"], z[f"in_{i}_t"], ts, te)
        assert np.array_equal(y, z[f"out_{i}_y"])
        assert [nt, dt, shift] == z[f"out_{i}_meta"].tolist()
    with pytest.raises(Exception):
        get_rf_inv_para(z["in_0_d"], z["in_0_t"], -100.0, 10.0)


# a checkout of the original RfSurfHmc project; its model/*.py are not part of this repository
REFERENCE = os.path.abspath(os.environ["RFSURFHMC_REFERENCE"]) if os.environ.get("RFSURFHMC_REFERENCE") else None


@pytest.mark.skipif(REFERENCE is None or not os.path.isdir(os.path.join(REFERENCE, "model")),
                    reason="needs the original RfSurfHmc project's model/*.py: set RFSURFHMC_REFERENCE to a checkout")
def test_references_unmodified_model_classes_run_over_the_dropin_stub_modules(oracle):
    """INTEGRATION.md §2: with `model/lib/libsurf.py` and `model/lib/librf.py` replaced by this repo's
    stub modules, the reference's UNMODIFIED model/*.py run.  So that no GPU is needed, the stubs'
    device context is replaced by an oracle-backed stand-in
    with the batched Context signatures, so what is checked is the binding itself: names, argument
    order, defaults, return tuples and shapes exactly as the reference's classes use them -- against
    the outputs of the same classes over the reference's own compiled modules (reference_code.npz)."""
    import importlib
    import sys
    import types
    from rfsurfhmc_b200 import _lib

    class OracleContext:
        """Context look-alike (batched drop-in signatures of rfsurfhmc_b200/_lib.py) on the CPU oracle"""

        def surf_forward(self, thk, vp, vs, rho, period, wavetype, mode=0, sphere=False):
            c, ok = oracle.surf_forward(thk, vp, vs, rho, period, wavetype, mode, sphere)
            return c[None, :], np.array([ok])

        def surf_adjoint_kernel(self, thk, vp, vs, rho, period, wavetype, mode=0, sphere=False, stale=True,
                                all_modes=False):
            r = oracle.surf_adjoint_kernel(thk, vp, vs, rho, period, wavetype, mode, sphere, stale)
            return tuple(a[None, ...] for a in r[:5]) + (np.array([r[5]]),)

        def rf_forward(self, *a, **k):
            return oracle.rf_forward(*a, **k)[None, :]

        def rf_kernel(self, *a, **k):
            rf, d = oracle.rf_kernel(*a, **k)
            return rf[None, :], d[None, ...]

        def rf_kernel_all(self, *a, **k):
            rf, d = oracle.rf_kernel_all(*a, **k)
            return rf[None, :], d[None, ...]

    saved_ctx = dict(_lib._default_ctx)
    saved_mods = {k: sys.modules.get(k) for k in ("model", "model.lib", "model.lib.libsurf", "model.lib.librf",
                                                  "model.model_surf", "model.model_rf",
                                                  "model.model_rf_swd_vs_thk")}
    sys.path.insert(0, REFERENCE)
    try:
        _lib._default_ctx[0] = OracleContext()
        stubs = importlib.import_module("rfsurfhmc_b200.model.lib")
        pkg = types.ModuleType("model")
        pkg.__path__ = [os.path.join(REFERENCE, "model")]  # the reference's own model/*.py ...
        sys.modules["model"] = pkg
        sys.modules["model.lib"] = stubs                  # ... over THIS repo's model/lib stub modules
        sys.modules["model.lib.libsurf"] = importlib.import_module("rfsurfhmc_b200.model.lib.libsurf")
        sys.modules["model.lib.librf"] = importlib.import_module("rfsurfhmc_b200.model.lib.librf")
        for m in ("model.model_surf", "model.model_rf", "model.model_rf_swd_vs_thk"):
            sys.modules.pop(m, None)
        RSurf = importlib.import_module("model.model_surf").SurfWD
        RRf = importlib.import_module("model.model_rf").ReceiverFunc
        RJoint = importlib.import_module("model.model_rf_swd_vs_thk").Joint_RF_SWD
        assert RSurf.__module__ == "model.model_surf"
        assert sys.modules["model.model_surf"].__file__.startswith(os.path.join(REFERENCE, "model") + os.sep)
        z = _ref_python_golden()
        cfg = f1_config()
        swd = RSurf(tRc=cfg["tRc"], tRg=cfg["tRg"])
        rf = RRf(cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], "P", "freq")
        joint = RJoint(1.0, 1.0, rf, swd)
        joint.set_obsdata(z["dobs"][:125], z["dobs"][125:])
        for i in range(3):
            U, g, d, f = joint.misfit_and_grad(z["glue_X"][i])
            assert f == bool(z["glue_flag"][i])
            assert np.isclose(U, z["glue_U"][i], rtol=1e-12)
            assert np.allclose(g, z["glue_grad"][i], rtol=1e-10, atol=1e-12 * np.abs(z["glue_grad"][i]).max())
            assert np.allclose(d, z["glue_dsyn"][i], rtol=1e-13, atol=1e-15)
        drf, dsw, flag = joint.forward(z["x_true"])
        assert drf.shape == (125,) and dsw.shape == (72,) and flag
    finally:
        sys.path.remove(REFERENCE)
        _lib._default_ctx.clear()
        _lib._default_ctx.update(saved_ctx)
        for k, v in saved_mods.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
