"""GPU parity tests proper: the sm_100a path called through the C ABI vs the CPU oracle and the
committed golden vectors.  Tolerances are BASELINE.json's: c, U <= 1e-6 relative; RF <= 1e-5 of the
trace peak; gradients <= 1e-4 relative (to the largest component of that gradient)."""
import os
import numpy as np
import pytest
from oracle.oracle import brocher
from rfsurfhmc_b200.fixtures import (f1_config, f1_true_model, driver_bounds, sorted_uniform_models,
                                     perturbed_models)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
TOL_C, TOL_RF, TOL_G = 1e-6, 1e-5, 1e-4


def rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def test_native_library_is_loaded(ctx):
    # the CUDA extension is the thing that runs: it is mapped into this process
    maps = open("/proc/self/maps").read()
    assert "librfsurf_b200.so" in maps
    l0 = ctx.launches
    ctx.surf_forward([5., 0.], [5., 6.], [3., 3.5], [2.5, 2.8], [5.], "Rc")
    assert ctx.launches > l0


def test_constant_bank_math_is_bit_identical_to_the_cuda_library(ctx):
    """The root search replaces exp / sincos / rsqrt by versions whose coefficients are constant-bank
    operands (fewer issue slots); the phase velocities only stay bit-identical to the previous build
    -- and as close to the oracle -- if these reproduce the CUDA library bit for bit."""
    assert ctx.selftest_math(1 << 22) == [0, 0, 0, 0, 0, 0]


def test_libsurf_dropin_vs_golden(ctx):
    g = np.load(os.path.join(G, "f1_dropin.npz"))
    thk, vs, vp, rho, T = g["thk"], g["vs"], g["vp"], g["rho"], g["T"]
    from rfsurfhmc_b200.model.lib import libsurf
    for wt in ("Rc", "Rg", "Lc", "Lg"):
        for mode in (0, 1, 2):
            c, ok = libsurf.forward(thk, vp, vs, rho, T, wt, mode)
            ref = g[f"fwd_{wt}_{mode}"]
            assert ok == bool(g[f"fwd_{wt}_{mode}_ok"])
            assert c.shape == (36,) and c.dtype == np.float64
            # missing higher modes: zeros (phase) / NaN (group) exactly where the reference has them
            assert np.array_equal(ref == 0, c == 0) and np.array_equal(np.isnan(ref), np.isnan(c))
            m = np.isfinite(ref) & (ref != 0)
            assert rel(c[m], ref[m]) <= TOL_C, (wt, mode)
        c, da, db, dr, dh, ok = libsurf.adjoint_kernel(thk, vp, vs, rho, T, wt)
        assert ok and da.shape == (36, 7)
        assert rel(c, g[f"ker_{wt}_c"]) <= TOL_C
        for got, key in ((da, "da"), (db, "db"), (dr, "dr"), (dh, "dh")):
            ref = g[f"ker_{wt}_{key}"]
            s = np.max(np.abs(ref))
            if s > 0:
                assert np.max(np.abs(got - ref)) / s <= TOL_G, (wt, key)
            else:
                assert np.all(got == 0)


def test_librf_dropin_vs_golden(ctx):
    g = np.load(os.path.join(G, "f1_dropin.npz"))
    thk, vs, vp, rho = g["thk"], g["vs"], g["vp"], g["rho"]
    q = thk * 0 + 9999.
    from rfsurfhmc_b200.model.lib import librf
    for rft in ("P", "S"):
        a = (thk, rho, vp, vs, q, q, 0.045, 125, 0.4, 1.5, 5.0, "freq", 0.001, rft)
        rf = librf.forward(*a)
        rf2, kl = librf.kernel_all(*a)
        peak = np.max(np.abs(g[f"rf_{rft}"]))
        assert rf.shape == (125,) and kl.shape == (4, 7, 125)
        assert np.max(np.abs(rf - g[f"rf_{rft}"])) <= TOL_RF * peak
        assert np.max(np.abs(rf2 - g[f"rf_{rft}"])) <= TOL_RF * peak
        ref = g[f"rf_{rft}_kl"]
        for ip in range(4):
            assert np.max(np.abs(kl[ip] - ref[ip])) <= TOL_G * np.max(np.abs(ref[ip]))
        for ip, nm in enumerate(("rho", "vp", "vs", "h")):
            _, k1 = librf.kernel(*a, par_type=nm)
            assert np.max(np.abs(k1 - ref[ip])) <= TOL_G * np.max(np.abs(ref[ip]))
    # F2 parameter set of the reference's test_forward.py (freq variant; nt=500 -> nft=512)
    vs2 = g["f2_vs"]
    vp2, rho2 = brocher(vs2)
    rf = librf.forward(thk, rho2, vp2, vs2, q, q, 0.045, 500, 0.1, 1.0, 5.0, "freq", 0.001, "P")
    assert np.max(np.abs(rf - g["f2_rf_freq"])) <= TOL_RF * np.max(np.abs(g["f2_rf_freq"]))


def test_dropins_vs_the_references_own_compiled_modules(ctx):
    """Same calls as the reference's pybind11 modules answered in tests/golden/reference_code.npz
    (src/SWD/main.cpp + surfdisp.cpp and src/RF/main.cpp compiled in place, Fortran entry points
    forwarded to the restated routines): every wave type x modes 0-2 x flat / spherical earth for
    four models, RF forward / kernel / kernel_all for both methods and both types."""
    z = np.load(os.path.join(G, "reference_code.npz"))
    from rfsurfhmc_b200.model.lib import libsurf, librf
    T = z["cpp_T"]
    n = 0
    for im, (h, a, v, r) in enumerate(z["cpp_models"]):
        for wt in ("Rc", "Rg", "Lc", "Lg"):
            for mode in (0, 1, 2):
                for sph in (False, True):
                    key = f"cpp{im}_{wt}_{mode}_{int(sph)}"
                    if key + "_fwd" not in z.files:
                        continue
                    ref = z[key + "_fwd"]
                    c, ok = libsurf.forward(h, a, v, r, T, wt, mode, sph)
                    assert ok == bool(z[key + "_ok"][0]), key
                    assert np.array_equal(ref == 0, c == 0) and np.array_equal(np.isnan(ref), np.isnan(c)), key
                    m = np.isfinite(ref) & (ref != 0)
                    assert rel(c[m], ref[m]) <= TOL_C, key
                    k = libsurf.adjoint_kernel(h, a, v, r, T, wt, mode, sph)
                    assert k[5] == bool(z[key + "_ok"][1]), key
                    kc = z[key + "_kc"]
                    m = np.isfinite(kc) & (kc != 0)
                    assert rel(k[0][m], kc[m]) <= TOL_C, key
                    for got, nm in zip(k[1:5], ("da", "db", "dr", "dh")):
                        if key + "_k" + nm not in z.files:
                            continue
                        rk = z[key + "_k" + nm][m]
                        sc = np.max(np.abs(rk)) if rk.size else 0.0
                        if sc > 0 and np.isfinite(sc):
                            assert np.nanmax(np.abs(got[m] - rk)) / sc <= TOL_G, (key, nm)
                    n += 1
    assert n == 48
    thk, vp, vs, rho = z["cpp_models"][0]
    q = thk * 0 + 9999.
    for method in ("freq", "time"):
        for rft in ("P", "S"):
            key = f"cpprf_{method}_{rft}"
            a = (thk, rho, vp, vs, q, q, 0.045, 125, 0.4, 1.5, 5.0, method, 0.001, rft)
            ref = z[key + "_fwd"]
            peak = np.max(np.abs(ref))
            assert np.max(np.abs(librf.forward(*a) - ref)) <= TOL_RF * peak, key
            _, kl = librf.kernel_all(*a)
            tol = TOL_G if method == "freq" else 1e-3   # deconit picks spikes: nonlinear in rounding
            for ip in range(4):
                assert np.max(np.abs(kl[ip] - z[key + "_all"][ip])) <= tol * np.max(np.abs(z[key + "_all"][ip])), (key, ip)


def test_references_own_test_script_on_the_gpu(ctx):
    """The curves of the reference's test_forward.py (run unmodified for
    tests/golden/reference_code.npz): time-domain receiver function (nt=500, dt=0.1, a=1.0) and the
    Rayleigh phase / group dispersion of its model, through the reference-shaped Python classes."""
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    z = np.load(os.path.join(G, "reference_code.npz"))
    tRc = np.linspace(5, 40, 36)
    model_swd = SurfWD(tRc=tRc, tRg=tRc.copy())
    model_rf = ReceiverFunc(0.045, 500, 0.1, 1.0, 5.0, 0.001, 'P', "time")
    thk = np.array([6, 6, 13, 5, 10, 30, 0]); vs = np.array([3.2, 3.4, 3.46, 3.7, 3.9, 4.5, 4.7])
    model_swd.set_thk(thk)
    model_rf.set_thk(thk)
    model = Joint_RF_SWD(1.0, 1.0, model_rf, model_swd)
    drsyn, dssyn, flag = model.forward(np.hstack((vs, thk)))
    assert flag
    assert np.max(np.abs(drsyn - z["tf_rf"])) <= TOL_RF * np.max(np.abs(z["tf_rf"]))
    assert rel(dssyn[:36], z["tf_Rc"]) <= TOL_C and rel(dssyn[36:], z["tf_Rg"]) <= TOL_C


def test_gpu_against_from_scratch_physics(ctx):
    """No oracle and no reference code in this test: the CUDA path against tests/independent.py (one
    linear system of plane-wave potentials per frequency / trial velocity) on the reference's default
    model -- Rayleigh and Love phase velocities of modes 0 and 1, and the P receiver function."""
    from independent import rayleigh_secular, love_secular, surface_response
    from rfsurfhmc_b200.model.lib import libsurf, librf
    x0 = f1_true_model()
    vs, thk = x0[:7], x0[7:]
    vp, rho = brocher(vs)
    f32 = lambda a: np.float32(a).astype(float)

    def root(fun, c_guess, Tp, par, width=3e-4):
        lo, hi = c_guess * (1 - width), c_guess * (1 + width)
        d0 = fun(lo, Tp, *par)
        ph = d0 / abs(d0)
        f = lambda x: (fun(x, Tp, *par) / ph).real
        flo = f(lo)
        assert np.sign(flo) != np.sign(f(hi)), (c_guess, Tp)
        for _ in range(50):
            mid = 0.5 * (lo + hi)
            fm = f(mid)
            if np.sign(fm) == np.sign(flo):
                lo, flo = mid, fm
            else:
                hi = mid
        return 0.5 * (lo + hi)
    T = np.array([5., 8., 12., 20., 30., 40.])
    for wt, fun, par in (("Rc", rayleigh_secular, [f32(thk), f32(vp), f32(vs), f32(rho)]),
                         ("Lc", love_secular, [f32(thk), f32(vs), f32(rho)])):
        for mode in (0, 1):
            c, ok = libsurf.forward(thk, vp, vs, rho, T, wt, mode)
            assert ok
            for Tp, ck in zip(T, c):
                if ck != 0.0:
                    assert abs(root(fun, ck, Tp, par) - ck) < 1.5e-6 * ck, (wt, mode, Tp)
    q = thk * 0 + 9999.
    p, nt, dt, a, tshift = 0.045, 125, 0.4, 1.5, 5.0
    rf = librf.forward(thk, rho, vp, vs, q, q, p, nt, dt, a, tshift, "freq", 0.001, "P")
    nft = 128
    sigma = 4.0 / (nft * dt)
    qf = 1 + 1 / (8 * 9999.**2) + 1j / (2 * 9999.)
    H = np.array([np.divide(*surface_response(2 * np.pi * kf / (nft * dt) - 1j * sigma, p, thk, vp * qf, vs * qf, rho))
                  for kf in range(nft // 2 + 1)])
    wr = 2 * np.pi * np.arange(nft // 2 + 1) / (nft * dt)
    tr = np.fft.irfft(H * np.exp(-wr**2 / (4 * a * a)) * np.exp(-1j * wr * tshift), nft)[:nt] / dt \
        * np.exp(sigma * (np.arange(nt) * dt - tshift))
    assert np.max(np.abs(tr - rf)) <= 2e-6 * np.max(np.abs(rf))


def test_error_conventions(ctx):
    from rfsurfhmc_b200._lib import RfsError
    from rfsurfhmc_b200.model.lib import libsurf, librf
    thk, vs = np.array([5., 0.]), np.array([3., 3.5])
    vp, rho = brocher(vs)
    q = thk * 0 + 9999.
    with pytest.raises(ValueError):
        libsurf.forward(thk, vp, vs, rho, [5.], "Rx")
    with pytest.raises(ValueError):
        librf.forward(thk, rho, vp, vs, q, q, 0.05, 64, 0.2, 2.0, 3.0, "freq", 0.001, "Q")
    with pytest.raises(ValueError):
        librf.kernel(thk, rho, vp, vs, q, q, 0.05, 64, 0.2, 2.0, 3.0, "freq", 0.001, "P", "zz")
    with pytest.raises(RfsError):  # a fluid layer below the top is rejected loudly
        libsurf.forward(np.array([5., 5., 0.]), np.array([5., 1.5, 6.]), np.array([3., 0.0, 3.5]),
                        np.array([2.5, 1.0, 2.8]), [5.], "Rc")
    with pytest.raises(RfsError):  # descending periods are rejected (mode cut-off logic needs ascending)
        libsurf.forward(thk, vp, vs, rho, [8., 5.], "Rc")


def test_root_failure_flag_and_batch_edges(ctx, oracle):
    # a strong inversion on top of a slow half-space: no fundamental root below betmx at long period
    thk = np.array([2., 0.]); vs = np.array([4.5, 1.6])
    vp, rho = brocher(vs)
    T = np.array([1., 2., 30., 60.])
    c0, ok0 = oracle.surf_forward(thk, vp, vs, rho, T, "Rc")
    c1, ok1 = ctx.surf_forward(thk, vp, vs, rho, T, "Rc")
    assert ok0 == bool(ok1[0])
    assert np.array_equal(c0 == 0, c1[0] == 0)
    # ragged batch sizes incl. 1 and a non-multiple of the block size; models are independent
    x0 = f1_true_model()
    X = perturbed_models(x0, 131, seed=3)
    vs_b, thk_b = X[:, :7], X[:, 7:]
    vp_b, rho_b = brocher(vs_b)
    Tq = np.array([6., 11., 23.])
    cb, okb = ctx.surf_forward(thk_b, vp_b, vs_b, rho_b, Tq, "Rc")
    c1_, _ = ctx.surf_forward(thk_b[77], vp_b[77], vs_b[77], rho_b[77], Tq, "Rc")
    assert cb.shape == (131, 3) and np.array_equal(cb[77], c1_[0])
    co, _ = oracle.surf_forward(thk_b[5], vp_b[5], vs_b[5], rho_b[5], Tq, "Rc")
    assert rel(cb[5], co) <= TOL_C


def _joint_ctx(ctx, dobs, cfg):
    ctx.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"])
    ctx.config_rf(7, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                  cfg["rf_type"], cfg["method"])
    ctx.config_obs(dobs)


def test_fused_joint_vs_golden(ctx):
    g = np.load(os.path.join(G, "f1_joint.npz"))
    cfg = f1_config()
    _joint_ctx(ctx, g["dobs"], cfg)
    U, gr, d, f = ctx.misfit_grad_host(g["X"])
    assert np.array_equal(f, g["flag"])
    m = f
    peak = np.max(np.abs(g["dsyn"][m, :125]), axis=1, keepdims=True)
    assert np.max(np.abs(d[m, :125] - g["dsyn"][m, :125]) / peak) <= TOL_RF
    assert rel(d[m, 125:], g["dsyn"][m, 125:]) <= TOL_C
    gs = np.max(np.abs(g["grad"][m]), axis=1, keepdims=True)
    assert np.max(np.abs(gr[m] - g["grad"][m]) / gs) <= TOL_G
    assert np.max(np.abs(U[m] - g["U"][m]) / np.maximum(g["U"][m], 1e-12)) <= 1e-5


def test_fused_joint_vs_oracle_fresh_models_and_subproblems(ctx, oracle):
    cfg = f1_config()
    x0 = f1_true_model()
    dobs = np.load(os.path.join(G, "f1_joint.npz"))["dobs"]
    X = np.vstack((sorted_uniform_models(driver_bounds(x0), 160, seed=101),
                   perturbed_models(x0, 96, seed=102, rel=0.1)))
    _joint_ctx(ctx, dobs, cfg)
    U1, g1, d1, f1 = ctx.misfit_grad_host(X)
    U0, g0, d0, f0 = oracle.joint_batch(X, dobs, cfg, nthreads=8)
    assert np.array_equal(f0, f1)
    m = f0
    e_c = np.max(np.abs(d1[m, 125:] - d0[m, 125:]) / np.abs(d0[m, 125:]), axis=1)
    e_rf = np.max(np.abs(d1[m, :125] - d0[m, :125]), axis=1) / np.max(np.abs(d0[m, :125]), axis=1)
    e_g = np.max(np.abs(g1[m] - g0[m]), axis=1) / np.max(np.abs(g0[m]), axis=1)
    assert e_rf.max() <= TOL_RF
    # root search is chaotic at the 1e-16 level for a small fraction of strongly inverted models
    # (DESIGN.md "parity statistics"): every model must be close, >= 99 % within the tolerances
    assert np.mean(e_c <= TOL_C) >= 0.99 and np.mean(e_g <= TOL_G) >= 0.99
    assert e_c.max() < 1e-3 and e_g.max() < 1e-2
    # RF-only and SWD-only objectives (ReceiverFunc / SurfWD misfit_and_grad)
    for which, sl in ((1, slice(0, 125)), (2, slice(125, 197))):
        ctx.config_obs(dobs[sl])
        Ua, ga, da, fa = oracle.joint_batch(X[:64], dobs[sl], cfg, which=which, nthreads=8)
        Ub, gb, db, fb = ctx.misfit_grad_host(X[:64], which=which)
        assert np.array_equal(fa, fb)
        eg = np.max(np.abs(gb[fa] - ga[fa]), axis=1) / np.max(np.abs(ga[fa]), axis=1)
        assert np.mean(eg <= TOL_G) >= 0.98
    ctx.config_obs(dobs)


def test_reference_shaped_python_api(ctx, oracle):
    """SurfWD / ReceiverFunc / Joint_RF_SWD driven exactly like the reference drivers do."""
    import yaml
    from rfsurfhmc_b200.model.model_rf import ReceiverFunc
    from rfsurfhmc_b200.model.model_surf import SurfWD
    from rfsurfhmc_b200.model.model_rf_swd_vs_thk import Joint_RF_SWD
    param = yaml.safe_load(open(os.path.join(G, "f1_param.yaml")))
    swd = SurfWD.init(**param["swd"])
    rfm = ReceiverFunc.init(**param["rf"])
    x = f1_true_model()
    model = Joint_RF_SWD(1.0, 1.0, rfm, swd)
    drf, dsw, flag = model.forward(x)
    assert flag and drf.shape == (125,) and dsw.shape == (72,)
    dobs = np.hstack((drf, dsw))
    model.set_obsdata(dobs[:125], dobs[125:])
    U, g, d, fl = model.misfit_and_grad(x)
    assert fl and U < 1e-20 and np.max(np.abs(g)) < 1e-8
    x2 = x * 1.03
    U, g, d, fl = model.misfit_and_grad(x2)
    U0, g0, d0, f0 = oracle.joint_batch(x2[None, :], dobs, f1_config())
    assert abs(U - U0[0]) <= 1e-6 * U0[0] and np.max(np.abs(g - g0[0])) <= TOL_G * np.max(np.abs(g0[0]))
    Ur, gr, dr = rfm.misfit_and_grad(x2)
    Us, gs_, ds, fs = swd.misfit_and_grad(x2)
    assert np.isclose(U, Ur + (125 / 72) * Us, rtol=1e-9)
    assert np.allclose(g, gr + (125 / 72) * gs_, rtol=1e-7, atol=1e-12)
    # finite-difference check of the fused gradient on the RF part (analytic kernels)
    e = np.zeros(14); e[2] = 1e-5
    fd = (rfm.misfit_and_grad(x2 + e)[0] - rfm.misfit_and_grad(x2 - e)[0]) / 2e-5
    assert abs(fd - gr[2]) <= 1e-5 * max(1.0, abs(gr[2]))


def test_size_independent_properties_at_scale(ctx):
    """BASELINE config-2-like sizes (n=40, 60 periods): Euler homogeneity c = sum(vp dc/dvp + vs dc/dvs
    + h dc/dh) and density invariance for every (model, period), without the oracle."""
    rng = np.random.default_rng(2)
    n, B = 40, 512
    i = np.arange(n - 1)
    thk = np.hstack((0.5 + 0.1 * i, [0.0]))[None, :] * (1 + 0.1 * rng.uniform(-1, 1, (B, n)))
    thk[:, -1] = 0.0
    vs0 = 2.0 + 2.7 * (np.arange(n) / 39.0)**0.7
    vs = np.clip(vs0[None, :] * (1 + 0.04 * rng.standard_normal((B, n))), 1.5, 5.0)
    vp, rho = brocher(vs)
    T = np.geomspace(2, 100, 60)
    for wt in ("Rc", "Lc"):
        c, da, db, dr, dh, ok = ctx.surf_adjoint_kernel(thk, vp, vs, rho, T, wt)
        assert ok.all()
        v32 = lambda a: a.astype(np.float32).astype(np.float64)
        euler = ((da * v32(vp)[:, None, :]).sum(2) + (db * v32(vs)[:, None, :]).sum(2) +
                 (dh * v32(thk)[:, None, :]).sum(2))
        assert np.max(np.abs(euler - c) / c) < 1e-4, wt  # kernels are evaluated at the f32-rounded, nevill-biased root
        assert np.max(np.abs((dr * v32(rho)[:, None, :]).sum(2))) < 3e-4, wt
    # all modes at once: higher modes are faster, missing ones are zeros at the long-period end
    c, *_ = ctx.surf_adjoint_kernel(thk[:64], vp[:64], vs[:64], rho[:64], T, "Rc", mode=2, all_modes=True)
    assert c.shape == (64, 3, 60)
    both = (c[:, 0] > 0) & (c[:, 1] > 0)
    assert np.all(c[:, 1][both] > c[:, 0][both])
    assert np.all((c[:, 2] == 0).sum(1) >= (c[:, 1] == 0).sum(1))


def test_time_domain_method_vs_oracle(ctx, oracle):
    """method="time" (iterative deconvolution, deconit.f90): forward trace, Frechet traces and the
    fused misfit+gradient.  The GPU keeps the spike train in the frequency domain (1 FFT/iteration
    instead of 8), so agreement is at rounding level, not bitwise."""
    g = np.load(os.path.join(G, "f1_dropin.npz"))
    thk, q = g["thk"], g["thk"] * 0 + 9999.
    vs2 = g["f2_vs"]
    vp2, rho2 = brocher(vs2)
    from rfsurfhmc_b200.model.lib import librf
    # F2 "smoke-time" fixture of the reference's test_forward.py (nt=500, dt=0.1, gauss=1)
    rf = librf.forward(thk, rho2, vp2, vs2, q, q, 0.045, 500, 0.1, 1.0, 5.0, "time", 0.001, "P")
    ref = g["f2_rf_time"]
    assert np.max(np.abs(rf - ref)) <= TOL_RF * np.max(np.abs(ref))
    # kernels on the F1 model with a short trace
    vs, vp, rho = g["vs"], g["vp"], g["rho"]
    a = (thk, rho, vp, vs, q, q, 0.045, 125, 0.4, 1.5, 5.0, "time", 0.001, "P")
    rf0, kl0 = oracle.rf_kernel_all(*a)
    rf1, kl1 = librf.kernel_all(*a)
    assert np.max(np.abs(rf1 - rf0)) <= TOL_RF * np.max(np.abs(rf0))
    for ip in range(4):
        s = np.max(np.abs(kl0[ip]))
        assert np.max(np.abs(kl1[ip] - kl0[ip])) <= TOL_G * s, ip
    _, k1 = librf.kernel(*a, par_type="vs")
    _, k0 = oracle.rf_kernel(*a, par_type="vs")
    assert np.max(np.abs(k1 - k0)) <= TOL_G * np.max(np.abs(k0))
    # fused RF objective with the time method
    cfg = dict(f1_config(), method="time")
    x0 = f1_true_model()
    X = perturbed_models(x0, 24, seed=9, rel=0.05)
    dobs = rf0
    ctx.config_rf(7, 0.045, 125, 0.4, 1.5, 5.0, 0.001, "P", "time")
    ctx.config_obs(dobs)
    Ub, gb, db, fb = ctx.misfit_grad_host(X, which=1)
    Ua, ga, da, fa = oracle.joint_batch(X, dobs, cfg, which=1, nthreads=8)
    assert np.max(np.abs(db - da)) <= TOL_RF * np.max(np.abs(da))
    eg = np.max(np.abs(gb - ga), axis=1) / np.max(np.abs(ga), axis=1)
    assert np.mean(eg <= TOL_G) >= 0.9 and eg.max() < 5e-2   # argmax spike picking can flip on near-ties


def test_spherical_earth_vs_oracle(ctx, oracle):
    """sphere=True: earth-flattening transformation (surfdisp96 `sphere`, bldsph, sprayl/splove,
    _flat2sphere, spherical branches of sregnpu/slegnpu), drop-ins and fused objective."""
    g = np.load(os.path.join(G, "f1_dropin.npz"))
    thk, vs, vp, rho = g["thk"], g["vs"], g["vp"], g["rho"]
    T = np.array([5., 8., 12., 20., 30., 40., 60.])
    from rfsurfhmc_b200.model.lib import libsurf
    for wt in ("Rc", "Rg", "Lc", "Lg"):
        c0, ok0 = oracle.surf_forward(thk, vp, vs, rho, T, wt, 0, True)
        c1, ok1 = libsurf.forward(thk, vp, vs, rho, T, wt, 0, True)
        assert ok0 == ok1 and rel(c1, c0) <= TOL_C, wt
        r0 = oracle.surf_adjoint_kernel(thk, vp, vs, rho, T, wt, 0, True)
        r1 = libsurf.adjoint_kernel(thk, vp, vs, rho, T, wt, 0, True)
        assert rel(r1[0], r0[0]) <= TOL_C, wt
        for i in range(1, 5):
            s = np.max(np.abs(r0[i]))
            if s > 0:
                assert np.max(np.abs(r1[i] - r0[i])) / s <= TOL_G, (wt, i)
    # sphericity raises long-period phase velocities by a fraction of a percent
    cf, _ = libsurf.forward(thk, vp, vs, rho, T, "Rc", 0, False)
    cs, _ = libsurf.forward(thk, vp, vs, rho, T, "Rc", 0, True)
    d = (cs - cf) / cf
    assert np.all(np.abs(d) < 0.02) and abs(d[-1]) > abs(d[0])
    # fused SWD objective on a spherical earth
    cfg = dict(f1_config(), sphere=True)
    x0 = f1_true_model()
    X = perturbed_models(x0, 32, seed=21, rel=0.05)
    dsw = np.hstack((oracle.surf_forward(thk, vp, vs, rho, cfg["tRc"], "Rc", 0, True)[0],
                     oracle.surf_forward(thk, vp, vs, rho, cfg["tRg"], "Rg", 0, True)[0]))
    ctx.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"], sphere=True)
    ctx.config_obs(dsw)
    Ub, gb, db, fb = ctx.misfit_grad_host(X, which=2)
    Ua, ga, da, fa = oracle.joint_batch(X, dsw, cfg, which=2, nthreads=8)
    assert np.array_equal(fa, fb)
    assert rel(db[fa], da[fa]) <= TOL_C
    eg = np.max(np.abs(gb[fa] - ga[fa]), axis=1) / np.max(np.abs(ga[fa]), axis=1)
    assert eg.max() <= TOL_G
    ctx.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"], sphere=False)


def test_forty_layer_models_vs_oracle(ctx, oracle):
    """BASELINE config-2/3 layer count (n=40 -> the NMAX=48 kernel instantiations): fused SWD objective
    with all four wave types and first higher mode, and fused RF objective, against the oracle."""
    rng = np.random.default_rng(7)
    n, B = 40, 12
    i = np.arange(n - 1)
    thk = np.hstack((0.5 + 0.1 * i, [0.0]))[None, :] * (1 + 0.1 * rng.uniform(-1, 1, (B, n)))
    thk[:, -1] = 0.0
    vs0 = 2.0 + 2.7 * (np.arange(n) / 39.0)**0.7
    vs = np.clip(vs0[None, :] * (1 + 0.04 * rng.standard_normal((B, n))), 1.5, 5.0)
    X = np.hstack((vs, thk))
    T = np.geomspace(2, 100, 24)
    base = dict(f1_config(), tRc=T, tRg=T, tLc=T, tLg=T, nt=256, dt=0.1, gauss=2.5, ray_p=0.06)
    for mode in (0, 1):
        cfg = dict(base, mode=mode)
        dobs = np.full(96, 3.2)
        ctx.config_swd(n, T, T, T, T, mode=mode)
        ctx.config_obs(dobs)
        Ub, gb, db, fb = ctx.misfit_grad_host(X, which=2)
        Ua, ga, da, fa = oracle.joint_batch(X, dobs, cfg, which=2, nthreads=8)
        assert np.array_equal(fa, fb)
        ok = np.isfinite(da) & (da != 0)
        assert np.array_equal(np.isfinite(db) & (db != 0), ok)       # same missing-mode pattern
        assert rel(db[ok], da[ok]) <= TOL_C
        fin = np.isfinite(ga).all(axis=1)
        assert np.array_equal(fin, np.isfinite(gb).all(axis=1))      # NaN gradients where a mode is missing
        if fin.any():
            eg = np.max(np.abs(gb[fin] - ga[fin]), axis=1) / np.max(np.abs(ga[fin]), axis=1)
            assert eg.max() <= TOL_G
    for rft in ("P", "S"):
        cfg = dict(base, rf_type=rft)
        ctx.config_rf(n, 0.06, 256, 0.1, 2.5, 5.0, 0.001, rft, "freq")
        dobs = np.zeros(256)
        ctx.config_obs(dobs)
        Ub, gb, db, fb = ctx.misfit_grad_host(X, which=1)
        Ua, ga, da, fa = oracle.joint_batch(X, dobs, cfg, which=1, nthreads=8)
        assert np.max(np.abs(db - da)) <= TOL_RF * np.max(np.abs(da))
        eg = np.max(np.abs(gb - ga), axis=1) / np.max(np.abs(ga), axis=1)
        assert eg.max() <= TOL_G, rft


def test_water_layer_on_top_vs_oracle(ctx, oracle):
    """Ocean model: fluid top layer (vs = 0): root search with the water-layer term of dltar4, fluid
    branches of the Rayleigh eigen kernels, Love ignoring the fluid; plus the scaling identities."""
    thk = np.array([3.0, 2.0, 5.0, 12.0, 0.0])
    vs = np.array([0.0, 2.2, 3.3, 3.9, 4.6])
    vp = np.array([1.5, 4.2, 5.9, 6.8, 8.1])
    rho = np.array([1.03, 2.3, 2.7, 2.9, 3.3])
    T = np.array([6., 10., 15., 25., 40.])
    from rfsurfhmc_b200.model.lib import libsurf
    for wt in ("Rc", "Rg", "Lc", "Lg"):
        c0, ok0 = oracle.surf_forward(thk, vp, vs, rho, T, wt)
        c1, ok1 = libsurf.forward(thk, vp, vs, rho, T, wt)
        assert ok0 == ok1 and rel(c1, c0) <= TOL_C, wt
        r0 = oracle.surf_adjoint_kernel(thk, vp, vs, rho, T, wt)
        r1 = libsurf.adjoint_kernel(thk, vp, vs, rho, T, wt)
        assert rel(r1[0], r0[0]) <= TOL_C, wt
        for i in range(1, 5):
            s = np.max(np.abs(r0[i]))
            if s > 0:
                assert np.max(np.abs(r1[i] - r0[i])) / s <= TOL_G, (wt, i)
    c, da, db, dr, dh, ok = libsurf.adjoint_kernel(thk, vp, vs, rho, T, "Rc")
    v32 = lambda a: a.astype(np.float32).astype(np.float64)
    euler = (da * v32(vp)).sum(1) + (db * v32(vs)).sum(1) + (dh * v32(thk)).sum(1)
    assert np.max(np.abs(euler - c) / c) < 1e-4       # homogeneity incl. the water layer's vp and h
    assert np.max(np.abs((dr * v32(rho)).sum(1))) < 3e-4
    assert np.all(db[:, 0] == 0.0)


def test_chunked_batches_give_identical_results(oracle):
    """Batches that exceed the workspace budget are processed in chunks inside the ABI: force a tiny
    budget and compare with the unchunked evaluation (bitwise: same kernels, same per-model work)."""
    import subprocess, sys, json
    code = r"""
import sys, os, json, numpy as np
sys.path.insert(0, %r)
from rfsurfhmc_b200._lib import Context
from rfsurfhmc_b200.fixtures import *
cfg = f1_config(); x0 = f1_true_model()
X = sorted_uniform_models(driver_bounds(x0), 777, seed=5)
dobs = np.load(os.path.join(%r, "f1_joint.npz"))["dobs"]
ctx = Context(0)
ctx.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"]); ctx.config_rf(7, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], cfg["rf_type"], cfg["method"]); ctx.config_obs(dobs)
U, g, d, f = ctx.misfit_grad_host(X)
np.savez(sys.argv[1], U=U, g=g, d=d, f=f)
"""
    import tempfile
    outs = []
    for budget in ("", "4"):
        with tempfile.NamedTemporaryFile(suffix=".npz", delete=False) as tf:
            env = dict(os.environ)
            if budget:
                env["RFS_WS_BUDGET_MB"] = budget       # 4 MiB -> ~100 models per chunk
            r = subprocess.run([sys.executable, "-c", code % (ROOT, G), tf.name], env=env,
                               capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stderr[-1500:]
            outs.append(dict(np.load(tf.name)))
    a, b = outs
    assert np.array_equal(a["f"], b["f"]) and np.array_equal(a["U"], b["U"])
    assert np.array_equal(a["g"], b["g"]) and np.array_equal(a["d"], b["d"])


def test_two_hundred_layer_models_vs_oracle(ctx, oracle):
    """BASELINE config-5 layer count (n=200 -> the NMAX=208 instantiations), joint objective."""
    rng = np.random.default_rng(11)
    n, B = 200, 3
    thk = 0.4 * (1 + 0.1 * rng.uniform(-1, 1, (B, n)))
    thk[:, -1] = 0.0
    vs0 = 2.0 + 2.7 * (np.arange(n) / (n - 1.0))**0.7
    vs = np.clip(vs0[None, :] * (1 + 0.02 * rng.standard_normal((B, n))), 1.5, 5.0)
    X = np.hstack((vs, thk))
    T = np.geomspace(1, 150, 12)
    cfg = dict(f1_config(), tRc=T, tRg=T, nt=128, dt=0.2, gauss=2.0, ray_p=0.05)
    dobs = np.hstack((np.zeros(128), np.full(24, 3.3)))
    ctx.config_swd(n, T, T)
    ctx.config_rf(n, 0.05, 128, 0.2, 2.0, 5.0, 0.001, "P", "freq")
    ctx.config_obs(dobs)
    Ub, gb, db, fb = ctx.misfit_grad_host(X)
    Ua, ga, da, fa = oracle.joint_batch(X, dobs, cfg, nthreads=3)
    assert np.array_equal(fa, fb) and fa.all()
    assert np.max(np.abs(db[:, :128] - da[:, :128])) <= TOL_RF * np.max(np.abs(da[:, :128]))
    assert rel(db[:, 128:], da[:, 128:]) <= TOL_C
    # a root can land exactly on a layer's S velocity after the float32 rounding (nu_b = 0): the
    # unfused-multiply oracle then divides by zero (NaN), FMA builds get a finite value.  Such
    # models are indeterminate in the reference too; compare the others.
    fin = np.isfinite(ga).all(axis=1)
    assert fin.sum() >= 2 and np.isfinite(gb).all()
    eg = np.max(np.abs(gb[fin] - ga[fin]), axis=1) / np.max(np.abs(ga[fin]), axis=1)
    assert eg.max() <= TOL_G


def test_host_pipeline_matches_blocking_api(ctx):
    """rfsurfhmc_b200.batched.HostPipeline (the e2e path of bench.py) returns, batch by batch, exactly
    what the blocking host API returns."""
    import torch
    from rfsurfhmc_b200.batched import HostPipeline
    cfg = f1_config()
    x0 = f1_true_model()
    dobs = np.load(os.path.join(G, "f1_joint.npz"))["dobs"]
    _joint_ctx(ctx, dobs, cfg)
    B = 96
    batches = [sorted_uniform_models(driver_bounds(x0), B, seed=300 + i) for i in range(5)]
    ref = [ctx.misfit_grad_host(X) for X in batches]
    pipe = HostPipeline(cfg, dobs, 7, B, device=0)
    got = []
    for X in batches:
        done = pipe.submit(torch.from_numpy(X).pin_memory())
        if done is not None:
            got.append([t.numpy().copy() for t in done])
    # two slots: the last two batches are still in flight
    pipe.slots[pipe.i % 2]["event"].synchronize()
    s = pipe.slots[pipe.i % 2]
    got.append([s[k].numpy().copy() for k in ("Uh", "Gh", "Dh", "Fh")])
    got.append([t.numpy().copy() for t in pipe.drain()])
    assert len(got) == 5
    for (U, g, d, f), (U2, g2, d2, f2) in zip(ref, got):
        assert np.array_equal(U, U2) and np.array_equal(g, g2) and np.array_equal(d, d2)
        assert np.array_equal(f, f2.astype(bool))


def test_bench_dump_outputs_is_the_last_timed_step(ctx, tmp_path):
    """`bench.py --dump-outputs DIR` writes what the last timed step returned.  With 6 timed steps over
    the 4 rotated input batches that is the second batch (a dump of any other step has other inputs),
    recomputed here through the blocking host API on the same seeded inputs and observations."""
    import subprocess, sys
    import bench
    B, steps = 256, 6
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                        "--chains", str(B), "--no-hmc", "--no-configs", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["U.npy", "dsyn.npy", "flag.npy", "grad.npy"]
    cfg, x0, _ = bench.workload(1, 0)
    _joint_ctx(ctx, np.zeros(197), cfg)
    ctx.config_obs(bench.make_dobs_gpu(ctx, cfg, x0))
    U, g, d, f = ctx.misfit_grad_host(bench.workload(B, 1000 + (steps - 1) % 4)[2])
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("U", "grad", "dsyn", "flag")}
    assert got["flag"].dtype == np.float32 and got["U"].dtype == np.float64
    assert got["U"].shape == (B,) and got["grad"].shape == (B, 14) and got["dsyn"].shape == (B, 197)
    assert np.array_equal(got["flag"] == 1, f) and f.sum() > B // 2
    for a, b in ((got["U"], U), (got["grad"], g), (got["dsyn"], d)):
        assert np.allclose(a[f], b[f], rtol=1e-12, atol=0)
