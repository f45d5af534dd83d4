"""Shape matrix of the CUDA path against the CPU oracle: every size-dependent dispatch choice runs here.

Layer counts: `nmax_for` (csrc/capi.cu) sends n to the NMAX = 8, 16, 48 or 208 instantiations of
swd_eigen_kernel and rf_propagate_kernel; the root search stages the model in shared memory only for
n <= RFS_ROOTS_STAGE_NMAX (8); pick_team has one threshold table for n <= 16 and another above.  The
matrix runs both sides of each bound, the bound itself (the local arrays full) and the documented
maximum of 208 layers, and checks that 1 and 209 layers are rejected.

Transform lengths: make_rf_cfg pads nt to nft = 2^lg, 2 <= nft <= 4096.  stockham_fft runs log4(nft/2)
radix-4 passes plus a radix-2 pass when log2(nft/2) is odd; decon_threads clamps to 64...512 threads and
time_threads to 64...256 (two butterflies per thread at nft = 4096).  The matrix runs every nft from 2 to
4096, each with nt = nft and nt = nft/2 + 1 where both exist.

rfs_profile_eval, the serialised copy of the fused evaluation that bench.py reads its per-kernel figures
from, must return the bits of rfs_misfit_grad_dev.

Tolerances are those of test_gpu_parity.py / test_gpu_sizes.py: c, U <= 1e-6 relative; RF <= 1e-5 of
the trace peak; gradients <= 1e-4 of the largest component.  The known exceptions get the allowances
those files grant, each stated where it is used."""
import ctypes
import os
import numpy as np
import pytest
from oracle.oracle import brocher
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, perturbed_models

pytestmark = pytest.mark.gpu
TOL_C, TOL_RF, TOL_G = 1e-6, 1e-5, 1e-4
NTH = os.cpu_count() or 8
RFS_E_ARG = -2
WAVES = ("Rc", "Rg", "Lc", "Lg")

# ---- layer-count matrix: both sides of every NMAX bound, the bounds themselves, the maximum
NS = [2, 3, 8, 9, 16, 17, 48, 49, 208]
DEPTH = 40.0                            # km above the half-space at every n: the same periods stay meaningful
T_SWD = np.geomspace(3.0, 60.0, 10)     # fundamental mode
T_HI = np.geomspace(1.5, 6.0, 6)        # first higher mode: short periods, where it exists
RF_N = dict(ray_p=0.06, nt=256, dt=0.15, gauss=2.5, time_shift=5.0, water=1e-3)

# ---- transform-length matrix (n = 7, the F1 model): every nft from 2 to 4096, nt = nft and nt = nft/2 + 1.
# nt = 1 is left out of the parity comparison: the reference pads with nextpow2(1) = 1 (a one-point
# transform), make_rf_cfg pads to nft = 2, so the damping sigma = 4 / (nft dt) and the transform differ and
# the two do not compute the same operation.
NTS = [2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128, 129, 256, 257, 512, 513, 1024, 1025, 2048, 2049, 4096]


def rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def grad_err(g1, g0):
    return np.max(np.abs(g1 - g0), axis=1) / np.max(np.abs(g0), axis=1)


def peak_err(a, b):
    """per row: largest difference over the reference trace's peak"""
    a, b = np.atleast_2d(a), np.atleast_2d(b)
    return np.max(np.abs(a - b), axis=1) / np.max(np.abs(b), axis=1)


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


@pytest.fixture(scope="module")
def sctx():
    """A context of this file's own: the root-search team and schedule overrides below cannot leak into
    other files' contexts."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from rfsurfhmc_b200._lib import Context
    c = Context(0)
    yield c
    c.close()


def models(B, n, seed, jitter=0.04):
    """test_gpu_sizes.layered with the thicknesses scaled to DEPTH km over the half-space at every n"""
    rng = np.random.default_rng(seed)
    thk0 = 0.5 + 0.1 * np.arange(n - 1)
    thk0 = np.hstack((thk0 * (DEPTH / thk0.sum()), [0.0]))
    thk = thk0[None, :] * (1 + 0.1 * rng.uniform(-1, 1, (B, n)))
    thk[:, -1] = 0.0
    vs0 = 2.0 + 2.7 * (np.arange(n) / (n - 1.0))**0.7
    vs = np.clip(vs0[None, :] * (1 + jitter * rng.standard_normal((B, n))), 1.5, 5.0)
    return np.hstack((vs, thk))


def batch(n):
    return 64 if n <= 17 else (16 if n <= 49 else 4)


def _split(X, n):
    vs, thk = X[:, :n], X[:, n:]
    vp, rho = brocher(vs)
    return thk, vp, vs, rho


def _rf_cfg(**kw):
    return dict(f1_config(), **RF_N, **kw)


# ------------------------------------------------------------------------------------ layer counts
@pytest.mark.parametrize("n", NS)
def test_swd_dropins_at_every_layer_count(sctx, oracle, n):
    """surf_adjoint_kernel (Rc, Rg, Lc, Lg; mode 0 and mode 1 on short periods; flat and spherical)
    against the oracle at every n of the matrix."""
    nmod = 4 if n <= 17 else (3 if n <= 49 else 2)
    X = models(nmod, n, 100 + n)
    thk, vp, vs, rho = _split(X, n)
    cut, indet = [], []
    errs = {nm: [] for nm in ("da", "db", "dr", "dh")}
    for sph in (False, True):
        for mode, T in ((0, T_SWD), (1, T_HI)):
            for wt in WAVES:
                c, da, db, dr, dh, ok = sctx.surf_adjoint_kernel(thk, vp, vs, rho, T, wt, mode=mode, sphere=sph)
                for b in range(nmod):
                    tag = (n, wt, mode, sph, b)
                    r0 = oracle.surf_adjoint_kernel(thk[b], vp[b], vs[b], rho[b], T, wt, mode, sph)
                    m0 = np.isfinite(r0[0]) & (r0[0] != 0)
                    m1 = np.isfinite(c[b]) & (c[b] != 0)
                    if mode == 0:
                        assert m0.all() and m1.all() and ok[b] and r0[5], tag
                    if not np.array_equal(m0, m1):
                        # a higher mode is cut off where its root reaches betmx (surfdisp96.f:483-487): a root
                        # within rounding of that limit exists in one build and not in the other
                        cut.append(tag)
                    else:
                        assert bool(ok[b]) == r0[5], tag
                    m = m0 & m1
                    if not m.any():
                        continue
                    assert rel(c[b][m], r0[0][m]) <= TOL_C, tag
                    ref = [k[m] for k in r0[1:5]]
                    if not all(np.isfinite(k).all() for k in ref):
                        # a float32-rounded root equal to a layer's vs (nu_b = 0): a division by zero in the
                        # unfused oracle, finite in FMA code (DESIGN.md §6)
                        indet.append(tag)
                        assert all(np.isfinite(k[b][m]).all() for k in (da, db, dr, dh)), tag
                        continue
                    # a higher mode within 1 % of the slowest layer's S velocity: nu_b ~ 0 in that layer, where
                    # the kernels are ill-conditioned in c
                    near = (mode > 0) & (np.abs(r0[0][m] / np.min(vs[b][vs[b] > 0]) - 1) < 1e-2)
                    for got, k0, nm in zip((da, db, dr, dh), ref, ("da", "db", "dr", "dh")):
                        s = np.max(np.abs(k0))
                        if s == 0:
                            assert np.all(got[b][m] == 0), tag + (nm,)
                            continue
                        e = np.max(np.abs(got[b][m] - k0), axis=1) / s    # per period, of the largest component
                        assert np.all(e[~near] <= TOL_G), tag + (nm, np.max(e[~near], initial=0))
                        # Near that S velocity the two builds' float32 roots differ within TOL_C (measured up to
                        # 8e-7) and the kernels follow them steeply: n = 2, mode 1, Rc / Rg at 1.5-3.4 s, phase or
                        # group velocity within 0.6 % of the 40 km layer's vs, measured up to 3.3e-2 in dr (8.4e-4
                        # in da).  Against central differences of an exact root of tests/independent.py (n = 2, Rc,
                        # mode 1, T = 1.98 s) dc/drho_0 is -3.08e-6, this build gives -3.10e-6, the oracle -3.58e-6.
                        assert np.all(e[near] <= 5e-2), tag + (nm, np.max(e[near], initial=0))
                        if not sph:
                            errs[nm].append(e[~near])
    # test_gpu_sizes.py grants max(2, B // 200) cut-off differences per mode and 0.5 % indeterminate models
    assert len(cut) <= 2, cut
    assert len(indet) <= 2, indet
    # The same root gives the same kernels to rounding: on a flat earth the median error per kernel type is
    # measured at 5e-15 (n = 2) to 2e-14 (n = 208) on a B200, so a kernel entry that is 1e-5 off for every
    # period (below TOL_G of the largest component) still fails here.
    for nm, e in errs.items():
        e = np.concatenate(e)
        assert e.size and np.median(e) <= 1e-10, (n, nm, np.median(e))


@pytest.mark.parametrize("n", NS)
def test_swd_objective_at_every_layer_count(sctx, oracle, n):
    """fused which = 2 objective (four wave types, mode 0): U, grad and dsyn against oracle.joint_batch"""
    B = batch(n)
    X = models(B, n, 200 + n)
    T = T_SWD
    dsw = np.full(4 * T.size, 3.3)
    sctx.config_swd(n, T, T, T, T)
    sctx.config_obs(dsw)
    Ub, gb, db, fb = sctx.misfit_grad_host(X, which=2)
    Ua, ga, da, fa = oracle.joint_batch(X, dsw, dict(f1_config(), tRc=T, tRg=T, tLc=T, tLg=T), which=2,
                                        nthreads=NTH)
    assert np.array_equal(fa, fb) and fa.all(), n
    assert rel(db, da) <= TOL_C, n
    # nu_b = 0 after the float32 rounding: NaN in the oracle, finite here (test_gpu_sizes.py C5 grants 3 of 32)
    fin = np.isfinite(ga).all(axis=1)
    assert (~fin).sum() <= max(1, B // 16) and np.isfinite(gb).all(), n
    eg = grad_err(gb[fin], ga[fin])
    assert eg.max() <= TOL_G, n
    # same roots, same kernels: the median is measured at 2e-15 (n = 2) to 6e-13 (n = 208) on a B200
    assert np.median(eg) <= 1e-9, (n, np.median(eg))
    assert rel(Ub[fin], Ua[fin]) <= 1e-5, n


@pytest.mark.parametrize("n", NS)
def test_root_mappings_bit_identical_at_every_layer_count(sctx, n):
    """thread mapping with the length-sorted job order on and off, the automatic choice and two team shapes:
    the same bits and the same number of secular evaluations at every n (staged and unstaged thread
    mapping, both pick_team tables).  Rayleigh and Love on different period lists, modes 0 and 1."""
    B = batch(n)
    X = models(B, n, 300 + n)
    sctx.config_swd(n, T_SWD, T_SWD, T_HI, T_HI, mode=[0, 1])
    sctx.config_obs(np.full(sctx.n_swd_data, 3.3))
    runs = {}
    try:
        for name, team, sched in (("thread", (0, 1), 0), ("thread-sorted", (0, 1), 1), ("auto", (-1, 1), -1),
                                  ("team16x2", (16, 2), -1), ("team32x4", (32, 4), -1)):
            sctx.set_roots_team(*team)
            sctx.set_roots_sched(sched)
            sctx.count_evals(True)
            out = sctx.misfit_grad_host(X, which=2)
            runs[name] = (out, sctx.read_evals())
            if team[0] >= 0:
                assert sctx.last_roots_team() == team, name
            assert sctx.last_roots_sched() == (sched == 1), name
    finally:
        sctx.count_evals(False)
        sctx.set_roots_team(-1)
        sctx.set_roots_sched(-1)
    ref, nev = runs["thread"]
    assert ref[3].any(), n
    for name, (out, ne) in runs.items():
        for nm, a, b in zip(("U", "grad", "dsyn", "flag"), ref, out):
            assert np.array_equal(a, b, equal_nan=True), (n, name, nm)
        assert ne == nev, (n, name, ne, nev)


@pytest.mark.parametrize("n", [9, 17])
def test_water_layer_on_top_through_nmax_16_and_48(sctx, oracle, n):
    """A fluid top layer (vs = 0) over n - 1 solid layers: the fluid branches of the root search and of the
    Rayleigh eigen kernels in the NMAX = 16 (n = 9) and NMAX = 48 (n = 17) instantiations."""
    nmod = 3
    S = models(nmod, n - 1, 400 + n)
    vs = np.hstack((np.zeros((nmod, 1)), S[:, :n - 1]))
    thk = np.hstack((np.full((nmod, 1), 3.0), S[:, n - 1:] * (37.0 / DEPTH)))
    vp, rho = brocher(vs)
    vp[:, 0], rho[:, 0] = 1.5, 1.03
    T = np.array([4., 6., 10., 15., 25., 40.])
    for wt in WAVES:
        c, da, db, dr, dh, ok = sctx.surf_adjoint_kernel(thk, vp, vs, rho, T, wt)
        for b in range(nmod):
            r0 = oracle.surf_adjoint_kernel(thk[b], vp[b], vs[b], rho[b], T, wt)
            assert bool(ok[b]) == r0[5] and r0[5], (n, wt, b)
            assert rel(c[b], r0[0]) <= TOL_C, (n, wt, b)
            for got, k0 in zip((da, db, dr, dh), r0[1:5]):
                s = np.max(np.abs(k0))
                if s > 0:
                    assert np.max(np.abs(got[b] - k0)) / s <= TOL_G, (n, wt, b)
            if wt[0] == "R":
                assert np.all(db[b][:, 0] == 0.0)     # no shear in the water


@pytest.mark.parametrize("n", NS)
def test_rf_at_every_layer_count(sctx, oracle, n):
    """RF forward (frequency and time method, P and S) against oracle.rf_forward at every n; the Frechet
    traces (rf_kernel_all) and the fused which = 1 objective against the oracle for n <= 49."""
    B = batch(n)
    X = models(B, n, 500 + n)
    nmod = min(B, 6)
    thk, vp, vs, rho = _split(X[:nmod], n)
    q = np.full_like(vs, 9999.)
    p, nt, dt, a, ts, wl = (RF_N[k] for k in ("ray_p", "nt", "dt", "gauss", "time_shift", "water"))
    for rft in ("P", "S"):
        for method in ("freq", "time"):
            rf1 = sctx.rf_forward(thk, rho, vp, vs, q, q, p, nt, dt, a, ts, method=method, water=wl, rf_type=rft)
            rf0 = np.array([oracle.rf_forward(thk[b], rho[b], vp[b], vs[b], q[b], q[b], p, nt, dt, a, ts,
                                              method=method, water=wl, rf_type=rft) for b in range(nmod)])
            assert peak_err(rf1, rf0).max() <= TOL_RF, (n, rft, method)
        if n > 49:
            continue   # the oracle's Frechet algorithm is O(n^2): n = 208 has its own gradient test below
        kw = dict(ray_p=p, nt=nt, dt=dt, gauss=a, time_shift=ts, water=wl, rf_type=rft, method="freq")
        r1, k1 = sctx.rf_kernel_all(thk[:2], rho[:2], vp[:2], vs[:2], q[:2], q[:2], **kw)
        for b in range(2):
            r0, k0 = oracle.rf_kernel_all(thk[b], rho[b], vp[b], vs[b], q[b], q[b], **kw)
            assert peak_err(r1[b], r0).max() <= TOL_RF, (n, rft)
            for i in range(4):
                # the frequency method has no root search: measured at 6e-14 at most on a B200 for n <= 49
                assert np.max(np.abs(k1[b, i] - k0[i])) <= 1e-9 * np.max(np.abs(k0[i])), (n, rft, i)
        Xr = X[:min(B, 16)]
        dobs = 0.02 * np.random.default_rng(n).standard_normal(nt)
        sctx.config_rf(n, p, nt, dt, a, ts, wl, rft, "freq")
        sctx.config_obs(dobs)
        Ub, gb, db, fb = sctx.misfit_grad_host(Xr, which=1)
        Ua, ga, da, fa = oracle.joint_batch(Xr, dobs, _rf_cfg(rf_type=rft), which=1, nthreads=NTH)
        assert fb.all() and peak_err(db, da).max() <= TOL_RF, (n, rft)
        # measured at 4e-13 at most on a B200 for n <= 49: a Frechet spectrum 1e-5 off fails
        assert rel(Ub, Ua) <= 1e-8 and grad_err(gb, ga).max() <= 1e-9, (n, rft)


@pytest.mark.parametrize("n", [n for n in NS if n <= 49])
def test_joint_objective_at_every_layer_count(sctx, oracle, n):
    """which = 0 (joint_assemble_kernel at each n): U, grad and dsyn against oracle.joint_batch"""
    B = min(batch(n), 32)
    X = models(B, n, 600 + n)
    T = T_SWD
    nt = RF_N["nt"]
    dobs = np.hstack((0.02 * np.random.default_rng(n).standard_normal(nt), np.full(4 * T.size, 3.3)))
    sctx.config_swd(n, T, T, T, T)
    sctx.config_rf(n, RF_N["ray_p"], nt, RF_N["dt"], RF_N["gauss"], RF_N["time_shift"], RF_N["water"], "P", "freq")
    sctx.config_obs(dobs)
    Ub, gb, db, fb = sctx.misfit_grad_host(X)
    Ua, ga, da, fa = oracle.joint_batch(X, dobs, _rf_cfg(tRc=T, tRg=T, tLc=T, tLg=T), nthreads=NTH)
    assert np.array_equal(fa, fb) and fa.all(), n
    assert peak_err(db[:, :nt], da[:, :nt]).max() <= TOL_RF, n
    assert rel(db[:, nt:], da[:, nt:]) <= TOL_C, n
    fin = np.isfinite(ga).all(axis=1)            # nu_b = 0 in the oracle, as in the SWD objective
    assert (~fin).sum() <= max(1, B // 16) and np.isfinite(gb).all(), n
    assert grad_err(gb[fin], ga[fin]).max() <= TOL_G, n
    assert rel(Ub[fin], Ua[fin]) <= 1e-5, n


def test_rf_gradient_at_208_layers_against_central_differences(sctx, oracle):
    """n = 208 (the documented maximum, NMAX = 208 full): the oracle's Frechet algorithm needs minutes per
    model here, so the fused which = 1 gradient is checked against the residual contracted with a Jacobian
    from central differences of oracle.rf_forward (the frequency method is smooth: a relative step of 1e-5
    gives about 1e-9 accuracy), on 12 parameters over the top, middle and bottom vs and thicknesses."""
    n, B = 208, 2
    X = models(B, n, 700)
    p, nt, dt, a, ts, wl = (RF_N[k] for k in ("ray_p", "nt", "dt", "gauss", "time_shift", "water"))
    q = np.full(n, 9999.)
    idx = [0, 1, 104, 206, 207, n + 0, n + 1, n + 103, n + 104, n + 205, n + 206, 105]

    def fwd(x, rft):
        vp, rho = brocher(x[:n])
        return oracle.rf_forward(x[n:], rho, vp, x[:n], q, q, p, nt, dt, a, ts, method="freq", water=wl,
                                 rf_type=rft)
    for rft in ("P", "S"):
        dobs = fwd(models(1, n, 701)[0], rft)
        sctx.config_rf(n, p, nt, dt, a, ts, wl, rft, "freq")
        sctx.config_obs(dobs)
        U, g, d, f = sctx.misfit_grad_host(X, which=1)
        assert f.all() and np.isfinite(g).all()
        for b in range(B):
            d0 = fwd(X[b], rft)
            assert peak_err(d[b], d0).max() <= TOL_RF, (rft, b)
            r = d[b] - dobs
            assert abs(U[b] - 0.5 * np.sum((d0 - dobs)**2)) <= 1e-6 * U[b], (rft, b)
            gs = np.max(np.abs(g[b]))
            for i in idx:
                h = 1e-5 * abs(X[b, i])
                xp, xm = X[b].copy(), X[b].copy()
                xp[i] += h
                xm[i] -= h
                fd = np.dot(r, (fwd(xp, rft) - fwd(xm, rft)) / (2 * h))
                assert abs(g[b, i] - fd) <= TOL_G * gs, (rft, b, i, g[b, i], fd)


def test_layer_counts_outside_the_instantiations_are_rejected(sctx):
    """n = 1 and n = 209 (above NMAX = 208): RFS_E_ARG from rfs_config_swd, rfs_config_rf,
    rfs_surf_forward and rfs_rf_forward, and a failed configuration call changes nothing
    (include/rfsurfhmc.h)."""
    from rfsurfhmc_b200._lib import RfsError
    cfg = f1_config()
    X = perturbed_models(f1_true_model(), 24, seed=5)
    sctx.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"])
    sctx.config_rf(7, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], "P", "freq")
    sctx.config_obs(np.full(125 + 72, 0.01))
    before = sctx.misfit_grad_host(X)
    L, h = sctx.L, sctx.h
    T = np.array([5., 10., 20.])
    for n in (1, 209):
        assert L.rfs_config_swd(h, n, 3, _dp(T), 3, _dp(T), 0, None, 0, None, 0, 0, 1) == RFS_E_ARG, n
        assert L.rfs_config_rf(h, n, 0.045, 125, 0.4, 1.5, 5.0, 0.001, 1, 1) == RFS_E_ARG, n
        Xn = models(2, max(n, 2), 9)[:, :n] if n > 1 else np.full((2, 1), 3.5)
        vs = Xn[:, :n]
        thk = np.full_like(vs, 0.2)
        thk[:, -1] = 0.0
        vp, rho = brocher(vs)
        with pytest.raises(RfsError) as e:
            sctx.surf_forward(thk, vp, vs, rho, T, "Rc")
        assert e.value.code == RFS_E_ARG, n
        with pytest.raises(RfsError) as e:
            sctx.rf_forward(thk, rho, vp, vs, thk * 0 + 9999., thk * 0 + 9999., 0.06, 64, 0.2, 2.0, 3.0, "freq")
        assert e.value.code == RFS_E_ARG, n
    after = sctx.misfit_grad_host(X)
    for a, b in zip(before, after):
        assert np.array_equal(a, b, equal_nan=True)


# -------------------------------------------------------------------------------- transform lengths
def _f1_rows(B=6, seed=31):
    X = perturbed_models(f1_true_model(), B, seed=seed, rel=0.05)
    X[0] = f1_true_model()
    return X


def _window(nt):
    """dt so that the trace spans the main conversions where nt allows it, the time shift inside the window"""
    dt = min(0.4, 50.0 / nt)
    return dt, min(5.0, 0.25 * nt * dt)


@pytest.mark.parametrize("nt", NTS)
def test_rf_frequency_method_at_every_transform_length(sctx, oracle, nt):
    """rf_forward, rf_kernel_all (rf_trace_kernel) and the fused which = 1 objective, P and S, against the
    oracle; the P forward also against the from-scratch plane-wave solution of tests/independent.py."""
    dt, ts = _window(nt)
    a, p, wl = 2.0, 0.045, 1e-3
    X = _f1_rows()
    thk, vp, vs, rho = _split(X, 7)
    q = np.full_like(vs, 9999.)
    for rft in ("P", "S"):
        kw = dict(nt=nt, dt=dt, gauss=a, time_shift=ts, water=wl, rf_type=rft, method="freq")
        rf1 = sctx.rf_forward(thk, rho, vp, vs, q, q, p, **kw)
        rf0 = np.array([oracle.rf_forward(thk[b], rho[b], vp[b], vs[b], q[b], q[b], p, **kw) for b in range(len(X))])
        assert peak_err(rf1, rf0).max() <= TOL_RF, (nt, rft)
        r1, k1 = sctx.rf_kernel_all(thk[:2], rho[:2], vp[:2], vs[:2], q[:2], q[:2], p, **kw)
        for b in range(2):
            r0, k0 = oracle.rf_kernel_all(thk[b], rho[b], vp[b], vs[b], q[b], q[b], p, **kw)
            assert peak_err(r1[b], r0).max() <= TOL_RF, (nt, rft)
            for i in range(4):
                assert np.max(np.abs(k1[b, i] - k0[i])) <= TOL_G * np.max(np.abs(k0[i])), (nt, rft, i)
        dobs = rf0[1] + 0.02 * np.random.default_rng(nt).standard_normal(nt)
        sctx.config_rf(7, p, nt, dt, a, ts, wl, rft, "freq")
        sctx.config_obs(dobs)
        Ub, gb, db, fb = sctx.misfit_grad_host(X, which=1)
        Ua, ga, da, fa = oracle.joint_batch(X, dobs, dict(f1_config(), ray_p=p, nt=nt, dt=dt, gauss=a, time_shift=ts,
                                                          water=wl, rf_type=rft), which=1, nthreads=NTH)
        assert fb.all() and peak_err(db, da).max() <= TOL_RF, (nt, rft)
        assert rel(Ub, Ua) <= 1e-8 and grad_err(gb, ga).max() <= TOL_G, (nt, rft)
    # independent float64 reference (test_gpu_parity.py's test_gpu_against_from_scratch_physics at every nft):
    # one linear system of plane-wave potentials per complex frequency, Gaussian, shift, inverse FFT, undamped
    from independent import surface_response
    nft = 1 << max(1, int(np.ceil(np.log2(nt))))
    sigma = 4.0 / (nft * dt)
    Q = 9999.
    qf = 1 + 1 / (8 * Q**2) + 1j / (2 * Q)
    H = np.array([np.divide(*surface_response(2 * np.pi * k / (nft * dt) - 1j * sigma, p, thk[0], vp[0] * qf,
                                              vs[0] * qf, rho[0])) for k in range(nft // 2 + 1)])
    wr = 2 * np.pi * np.arange(nft // 2 + 1) / (nft * dt)
    tr = np.fft.irfft(H * np.exp(-wr**2 / (4 * a * a)) * np.exp(-1j * wr * ts), nft)[:nt] / dt \
        * np.exp(sigma * (np.arange(nt) * dt - ts))
    rfp = sctx.rf_forward(thk[:1], rho[:1], vp[:1], vs[:1], q[:1], q[:1], p, nt, dt, a, ts, method="freq", water=wl,
                          rf_type="P")
    assert peak_err(rfp[0], tr).max() <= TOL_RF, nt


@pytest.mark.parametrize("nt", NTS)
def test_rf_time_method_at_every_transform_length(sctx, oracle, nt):
    """rf_time_kernel (one or two butterflies per thread, 64...256 threads): rf_forward, P and S, and the
    fused which = 1 objective against the oracle"""
    dt, ts = _window(nt)
    a, p, wl = 2.0, 0.045, 1e-3
    X = _f1_rows()
    thk, vp, vs, rho = _split(X, 7)
    q = np.full_like(vs, 9999.)
    for rft in ("P", "S"):
        kw = dict(nt=nt, dt=dt, gauss=a, time_shift=ts, water=wl, rf_type=rft, method="time")
        rf1 = sctx.rf_forward(thk, rho, vp, vs, q, q, p, **kw)
        rf0 = np.array([oracle.rf_forward(thk[b], rho[b], vp[b], vs[b], q[b], q[b], p, **kw) for b in range(len(X))])
        assert peak_err(rf1, rf0).max() <= TOL_RF, (nt, rft)
        Xf = _f1_rows(3, seed=32)
        dobs = rf0[0] + 0.02 * np.random.default_rng(nt).standard_normal(nt)
        sctx.config_rf(7, p, nt, dt, a, ts, wl, rft, "time")
        sctx.config_obs(dobs)
        Ub, gb, db, fb = sctx.misfit_grad_host(Xf, which=1)
        Ua, ga, da, fa = oracle.joint_batch(Xf, dobs, dict(f1_config(), ray_p=p, nt=nt, dt=dt, gauss=a, time_shift=ts,
                                                           water=wl, rf_type=rft, method="time"), which=1, nthreads=NTH)
        assert fb.all() and peak_err(db, da).max() <= TOL_RF, (nt, rft)
        # argmax spike picking in the Frechet traces can flip on near-ties (test_gpu_parity.py grants 10 % of
        # the models above TOL_G and 5e-2 at most); with three models here, one
        eg = grad_err(gb, ga)
        assert np.sum(eg > TOL_G) <= 1 and eg.max() < 5e-2, (nt, rft, eg.max())


def _width_passes(c, nt, dt, ts, widths, dobs, X):
    """one one-width configuration per width on the same context, in list order"""
    U, g, d = 0.0, 0.0, []
    for ig, a in enumerate(widths):
        c.config_rf(7, 0.045, nt, dt, float(a), ts, 1e-3, "P", "freq")
        c.config_obs(dobs[ig * nt:(ig + 1) * nt])
        Ui, gi, di, fi = c.misfit_grad_host(X, 1)
        assert fi.all()
        U, g = U + Ui, g + gi
        d.append(di)
    return U, g, np.hstack(d)


@pytest.mark.parametrize("nt,G", [(5, 3), (65, 3), (513, 3), (2049, 3), (4096, 16)])
def test_gauss_widths_at_transform_lengths(sctx, nt, G):
    """rf_decon_kernel<true> (several widths on one staged spectrum, the weight accumulator in shared
    memory): every trace equals its one-width pass bit for bit, misfit and gradient the sums over the
    passes (to 1e-12 and 1e-10, as test_gpu_rf_gauss.py checks).  16 widths is RFS_MAX_GAUSS."""
    dt, ts = _window(nt)
    widths = [1.0, 2.5, 5.0] if G == 3 else list(np.linspace(0.5, 8.0, G))
    X = _f1_rows(8, seed=33)
    dobs = 0.02 * np.random.default_rng(G + nt).standard_normal(G * nt)
    sctx.config_rf(7, 0.045, nt, dt, widths, ts, 1e-3, "P", "freq")
    sctx.config_obs(dobs)
    U, g, d, f = sctx.misfit_grad_host(X, 1)
    assert f.all() and d.shape == (len(X), G * nt) and np.isfinite(d).all()
    U0, g0, d0 = _width_passes(sctx, nt, dt, ts, widths, dobs, X)
    assert np.array_equal(d, d0), nt
    assert np.all(np.abs(U - U0) <= 1e-12 * np.abs(U0)), nt
    assert np.all(np.abs(g - g0) <= 1e-10 * np.abs(g0).max(axis=1, keepdims=True)), nt


def test_transform_lengths_outside_the_range_are_rejected(sctx):
    """nt = 0 and nt = 4097 (nft = 8192, above the 4096-point cap): RFS_E_ARG from the configuration and
    the drop-in"""
    from rfsurfhmc_b200._lib import RfsError
    x = f1_true_model()
    vs, thk = x[:7][None, :], x[7:][None, :]
    vp, rho = brocher(vs)
    q = np.full_like(vs, 9999.)
    for nt in (0, 4097):
        assert sctx.L.rfs_config_rf(sctx.h, 7, 0.045, nt, 0.01, 1.5, 5.0, 0.001, 1, 1) == RFS_E_ARG, nt
        for method in ("freq", "time"):
            with pytest.raises(RfsError) as e:
                sctx.rf_forward(thk, rho, vp, vs, q, q, 0.045, nt, 0.01, 1.5, 5.0, method=method)
            assert e.value.code == RFS_E_ARG, (nt, method)


# ------------------------------------------------------------------------ rfs_profile_eval
def _device_eval(c, X, which, profile):
    import torch
    dev = torch.device("cuda", c.device)
    x = torch.from_numpy(np.ascontiguousarray(X)).to(dev)
    B = len(X)
    U = torch.full((B,), -1.0, dtype=torch.float64, device=dev)
    g = torch.full_like(x, -1.0)
    d = torch.full((B, c.ndata(which)), -1.0, dtype=torch.float64, device=dev)
    f = torch.full((B,), 7, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev)
    torch.cuda.synchronize(dev)
    l0 = c.launches
    args = (B, x.data_ptr(), which, U.data_ptr(), g.data_ptr(), d.data_ptr(), f.data_ptr(), st.cuda_stream)
    prof = c.profile_eval(*args) if profile else c.misfit_grad_dev(*args)
    torch.cuda.synchronize(dev)
    return [t.cpu().numpy() for t in (U, g, d, f)], prof, c.launches - l0


def _joint_at(c, n, X_seed):
    T = T_SWD
    nt = RF_N["nt"]
    c.config_swd(n, T, T, T, T)
    c.config_rf(n, RF_N["ray_p"], nt, RF_N["dt"], RF_N["gauss"], RF_N["time_shift"], RF_N["water"], "P", "freq")
    c.config_obs(np.hstack((0.02 * np.random.default_rng(n).standard_normal(nt), np.full(4 * T.size, 3.3))))
    return models(96, n, X_seed), 0


def _time_4096(c):
    nt = 4096
    dt, ts = _window(nt)
    c.config_rf(7, 0.045, nt, dt, 2.0, ts, 1e-3, "P", "time")
    c.config_obs(0.02 * np.random.default_rng(4).standard_normal(nt))
    return _f1_rows(4, seed=34), 1


def _one_set(c):
    # rfs_profile_eval takes no set array: a context that holds several observation sets is out of its
    # reach (RFS_E_CONFIG).  One set given as an [1, ndata] table is the case it serves.
    cfg = f1_config()
    c.config_swd(7, tRc=cfg["tRc"], tRg=cfg["tRg"])
    c.config_rf(7, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], "P", "freq")
    c.config_obs(np.full((1, 125 + 72), 0.01))
    assert c.nsets == 1
    X = perturbed_models(f1_true_model(), 200, seed=35, rel=0.3)
    return X, 0


PROFILE_CASES = {"joint-n8": lambda c: _joint_at(c, 8, 800), "joint-n16": lambda c: _joint_at(c, 16, 816),
                 "time-nt4096": _time_4096, "one-set": _one_set}


@pytest.mark.parametrize("case", list(PROFILE_CASES))
def test_profile_eval_returns_the_bits_of_misfit_grad_dev(sctx, case):
    """rfs_profile_eval runs the fused evaluation with the RF branch serialised and CUDA events around
    every launch: U, grad, dsyn and flag must be the bits of rfs_misfit_grad_dev on the same inputs; every
    kernel class reports finite, non-negative milliseconds; and the per-class launch counts add up to the
    call's increase of rfs_launch_count (both count LAUNCH / LAUNCH_TU launches; the FFT twiddle kernel of
    run_rf_spectra is counted by neither)."""
    X, which = PROFILE_CASES[case](sctx)
    ref, _, nl_dev = _device_eval(sctx, X, which, False)
    got, prof, nl = _device_eval(sctx, X, which, True)
    for nm, a, b in zip(("U", "grad", "dsyn", "flag"), ref, got):
        assert np.array_equal(a, b, equal_nan=True), (case, nm)
    assert np.all(ref[3] <= 1) and ref[3].any(), case
    assert len(prof) == sctx.PROF_NK
    for k, (ms, cnt) in prof.items():
        assert np.isfinite(ms) and ms >= 0.0 and cnt >= 0, (case, k, ms, cnt)
        assert cnt > 0 or ms == 0.0, (case, k)
    assert sum(cnt for _, cnt in prof.values()) == nl, (case, prof, nl)
    assert nl > 0 and nl_dev > 0
    # the classes the evaluation runs are the ones reported
    assert prof["prep_models"][1] >= 1 and prof["rf_layer"][1] >= 1 and prof["rf_propagate"][1] >= 1, case
    if which == 0:
        assert prof["swd_roots"][1] >= 1 and prof["swd_eigen"][1] >= 1 and prof["assemble"][1] >= 1, case
        assert prof["rf_decon"][1] >= 1, case
    else:
        assert prof["rf_time_domain"][1] >= 1 and prof["swd_roots"][1] == 0, case
