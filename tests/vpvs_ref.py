"""Reference side of the [vs, thk, vpvs] parameterisation (include/rfsurfhmc.h: rfs_config_param), for
the tests only.

oracle/hmc_ref.py restates the reference samplers for x = [vs, thk] and stays as it is: it is pinned
against the reference's own code.  The device samples [vs, thk, vpvs] with one different step, the
initial model (vs sorted ascending, thk AND Vp/Vs permuted with it, every entry in its box except the
half-space thickness at index 2n - 1).  run_base / run_da below are hmc_ref's own functions, run with
that initial-model rule in place of hmc_ref._initial_model; everything else (mirror, leapfrog,
accept/reject, dual averaging, the NumPy-legacy random stream) is hmc_ref's code unchanged.

vpvs_objective composes the objective of [vs, thk, vpvs] from the oracle's per-field kernels, so that the
samplers' restatement and the parity tests have a reference for it."""
import types
import numpy as np
from oracle import hmc_ref


def initial_model(bounds, rs, npar=3):
    """hmc_ref._initial_model for npar parameter blocks of n layers: draws in the box until every entry
    but the half-space thickness (index 2n - 1) lies in it, vs sorted ascending and the other blocks
    permuted with it.  npar = 2 is hmc_ref's rule."""
    n2 = bounds.shape[0]
    n = n2 // npar
    while True:
        x = np.zeros(n2)
        for i in range(n2):
            x[i] = bounds[i, 0] + (bounds[i, 1] - bounds[i, 0]) * rs.rand()
        idx = np.argsort(x[:n])
        for j in range(npar):
            x[j * n:(j + 1) * n] = x[j * n:(j + 1) * n][idx]
        ok = all(not (x[i] < bounds[i, 0] or x[i] > bounds[i, 1]) for i in range(n2) if i != 2 * n - 1)
        if ok:
            return x


def _with_vpvs_start(fn):
    """hmc_ref's sampler function `fn` with initial_model as its initial-model step (same code object,
    globals where _initial_model is the three-block rule; hmc_ref itself is not modified)."""
    g = dict(vars(hmc_ref), _initial_model=initial_model)
    return types.FunctionType(fn.__code__, g, fn.__name__, fn.__defaults__, fn.__closure__)


run_base = _with_vpvs_start(hmc_ref.run_base)
run_da = _with_vpvs_start(hmc_ref.run_da)


_BR = (1.6612, -0.4721, 0.0671, -0.0043, 0.000106)


def vpvs_objective(O, x, dobs, cfg, which=0):
    """Objective of x = [vs(n), thk(n), k(n)] (vp = k vs, rho = Brocher's density of vp) composed from
    the oracle's per-field kernels: rf_kernel_all (d/d rho, vp, vs, h of each RF trace) and
    surf_adjoint_kernel (dc/d vp, vs, rho, h on the float32-cast model, as the device's SWD boundary).
    g_vs = K_b + k (K_a + drho/dvp K_r), g_thk = K_h, g_k = vs (K_a + drho/dvp K_r).
    cfg as Oracle.joint_batch, except that ray_p and gauss may be lists (RF data [ray][gauss][nt]) and
    mode an ascending list (SWD data [mode][Rc, Rg, Lc, Lg]).  Returns (U, grad [3n], dsyn, flag) with the
    failure convention (0, zeros, dobs, False) (SWD only: zeros for dsyn)."""
    x = np.asarray(x, dtype=np.float64)
    n = x.size // 3
    vs, thk, k = x[:n], x[n:2 * n], x[2 * n:]
    vp = k * vs
    rho = sum(c * vp**(i + 1) for i, c in enumerate(_BR))
    drda = sum(c * (i + 1) * vp**i for i, c in enumerate(_BR))
    dobs = np.asarray(dobs, dtype=np.float64)
    nt = int(cfg["nt"])
    rays, widths = np.atleast_1d(cfg["ray_p"]), np.atleast_1d(cfg["gauss"])
    n1 = nt * rays.size * widths.size if which != 2 else 0
    g_rf, g_sw = np.zeros(3 * n), np.zeros(3 * n)
    U_rf = U_sw = 0.0
    d = []

    def contract(res, ka, kb, kr, kh):
        # ka, kb, kr, kh [n][ndata]: sensitivities of the data to vp, vs, rho, thk of each layer
        ch = (ka + drda[:, None] * kr) @ res
        return np.concatenate((kb @ res + k * ch, kh @ res, vs * ch))

    if which != 2:
        q = np.full(n, 9999.)
        o = 0
        for p in rays:
            for w in widths:
                rf, K = O.rf_kernel_all(thk, rho, vp, vs, q, q, float(p), nt, float(cfg["dt"]), float(w),
                                        float(cfg["time_shift"]), cfg.get("method", "freq"),
                                        float(cfg.get("water", 0.001)), cfg.get("rf_type", "P"))
                res = rf - dobs[o:o + nt]
                U_rf += 0.5 * np.sum(res**2)
                g_rf += contract(res, K[1], K[2], K[0], K[3])
                d.append(rf)
                o += nt
    nsw = 0
    if which != 1:
        o = n1
        for mode in np.atleast_1d(cfg.get("mode", 0)):
            for wt in ("Rc", "Rg", "Lc", "Lg"):
                T = np.asarray(cfg.get("t" + wt, []), dtype=np.float64)
                if T.size == 0:
                    continue
                c, da, db, dr, dh, ok = O.surf_adjoint_kernel(thk, vp, vs, rho, T, wt, int(mode),
                                                              bool(cfg.get("sphere", False)),
                                                              bool(cfg.get("stale", True)))
                if not ok:
                    return 0.0, np.zeros(3 * n), (dobs if which == 0 else np.zeros(dobs.size)), False
                res = c - dobs[o:o + T.size]
                U_sw += 0.5 * np.sum(res**2)
                g_sw += contract(res, da.T, db.T, dr.T, dh.T)
                d.append(c)
                o += T.size
                nsw += T.size
    w = (float(cfg.get("sigma1", 1.0)) / float(cfg.get("sigma2", 1.0)))**2 * n1 / nsw if which == 0 else 1.0
    return U_rf + w * U_sw, g_rf + w * g_sw, np.concatenate(d), True


def oracle_vpvs_f(O, dobs, cfg, which=0):
    """misfit_and_grad callable of the [vs, thk, vpvs] objective (vpvs_objective), the counterpart of
    hmc_ref.oracle_joint_f for the samplers' restatement."""
    def f(x):
        return vpvs_objective(O, x, dobs, cfg, which)
    return f
