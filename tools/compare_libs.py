"""Bitwise comparison of two builds of librfsurf_b200.so on the same inputs (used to show that an
optimisation leaves every result bit unchanged).

    python tools/compare_libs.py build/base.so build/variant.so [--batch 8192]

Each library runs in its own process (RFS_LIB selects it).  Legs, each reported on its own line:
  joint_f1   U, grad, dsyn, flag of the F1 joint objective on realistic + wild models (one chunk)
  surf       the SWD drop-ins: Love/Rayleigh, n=40, modes 0..2
  time_rf    RF-only objective, time method, two rays x two Gaussian widths, three observation sets
             with a ray table and an RF sample mask, one set index per row
  time_joint the same as a joint objective
  time_chunk the same joint objective on a context created with RFS_WS_BUDGET_MB=1 (several chunks)
  librf      the librf drop-ins rf_forward (both methods, P and S) and rf_kernel_all (both methods)"""
import argparse, os, subprocess, sys, tempfile
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _time_sets(ctx, cfg, x0, B, which):
    """RF method "time", rays [0.04, 0.06] x widths [1.0, 2.5], S = 3 sets with a ray table and an RF
    sample mask; U, grad, dsyn, flag of `which` on B rows, row b on set b % 3."""
    from rfsurfhmc_b200 import fixtures as F
    n, S = x0.size // 2, 3
    ctx.config_swd(n, cfg["tRc"], cfg["tRg"], cfg["tLc"], cfg["tLg"], cfg["mode"], cfg["sphere"])
    ctx.config_rf(n, [0.04, 0.06], cfg["nt"], cfg["dt"], [1.0, 2.5], cfg["time_shift"], cfg["water"],
                  cfg["rf_type"], "time")
    rays = np.array([[0.040, 0.060], [0.042, 0.058], [0.045, 0.065]])
    use = np.ones((S, 2, 2, cfg["nt"]), dtype=bool)
    use[1, :, :, 100:] = False
    use[2, 1, 0] = False

    def tables(dobs):
        ctx.config_obs(dobs, [1.0, 0.5, 2.0], [1.0, 1.5, 0.8])
        ctx.config_obs_rays(rays)
        ctx.config_obs_rf_samples(use)

    sets0 = np.arange(S, dtype=np.int32)
    tables(np.zeros((S, ctx.ndata(which))))
    _, _, d0, _ = ctx.misfit_grad_host(F.perturbed_models(x0, S, 21, rel=0.05), which, sets=sets0)
    tables(d0 + 0.01 * np.random.default_rng(22).standard_normal(d0.shape))
    X = np.vstack((F.perturbed_models(x0, B - B // 4, 23, rel=0.1),
                   np.random.default_rng(24).uniform(0.5, 1.5, (B // 4, 2 * n)) * x0 + 0.01))
    return _masked(*ctx.misfit_grad_host(X, which, sets=np.arange(B, dtype=np.int32) % S))


def _masked(U, g, d, f):
    ok = f.astype(bool)   # models whose root search failed carry unspecified values: compare the rest
    return dict(U=np.where(ok, U, 0.0), g=np.where(ok[:, None], g, 0.0), d=np.where(ok[:, None], d, 0.0), f=f)


def worker(out, B):
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200 import fixtures as F
    cfg = F.f1_config()
    x0 = F.f1_true_model()
    n = x0.size // 2
    ctx = Context(0)
    ctx.config_swd(n, cfg["tRc"], cfg["tRg"], cfg["tLc"], cfg["tLg"], cfg["mode"], cfg["sphere"])
    ctx.config_rf(n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                  cfg["rf_type"], cfg["method"])
    nd = cfg["nt"] + 2 * len(cfg["tRc"])
    ctx.config_obs(np.zeros(nd))
    _, _, d0, _ = ctx.misfit_grad_host(x0[None, :])
    ctx.config_obs(d0[0])
    X = np.vstack((F.perturbed_models(x0, B // 2, 11, rel=0.1),
                   F.sorted_uniform_models(F.driver_bounds(x0), B // 2, 12),
                   np.random.default_rng(13).uniform(0.5, 1.5, (B // 2, 2 * n)) * x0 + 0.01))
    res = {f"joint_f1/{k}": v for k, v in _masked(*ctx.misfit_grad_host(X)).items()}
    # n=40, all four wave types, modes 0..2 through the drop-in
    rng = np.random.default_rng(5)
    nl, Bm = 40, 256
    thk = np.hstack((0.5 + 0.1 * np.arange(nl - 1), [0.0]))[None, :] * (1 + 0.1 * rng.uniform(-1, 1, (Bm, nl)))
    vs = np.clip((2.0 + 2.7 * (np.arange(nl) / (nl - 1.0))**0.7)[None, :] * (1 + 0.04 * rng.standard_normal((Bm, nl))), 1.5, 5.0)
    vp = 1.73 * vs
    rho = 0.32 * vp + 0.77
    T = np.geomspace(2, 100, 30)
    for wt in ("Rc", "Rg", "Lc", "Lg"):
        for mode in (0, 1, 2):
            o = ctx.surf_adjoint_kernel(thk, vp, vs, rho, T, wt, mode)
            for i, a in enumerate(o):
                res[f"surf/{wt}{mode}_{i}"] = np.asarray(a)
    Bt = max(B // 8, 8)
    for which, leg in ((1, "time_rf"), (0, "time_joint")):
        res.update({f"{leg}/{k}": v for k, v in _time_sets(ctx, cfg, x0, Bt, which).items()})
    os.environ["RFS_WS_BUDGET_MB"] = "1"   # read when the context is created
    chunked = Context(0)
    del os.environ["RFS_WS_BUDGET_MB"]
    res.update({f"time_chunk/{k}": v for k, v in _time_sets(chunked, cfg, x0, Bt, 0).items()})
    chunked.close()
    # librf drop-ins on the F1 layering
    Xl = F.perturbed_models(x0, 64, 31, rel=0.1)
    vs, thk = Xl[:, :n], Xl[:, n:]
    vp = 1.73 * vs
    rho = 0.32 * vp + 0.77
    q = np.full_like(vs, 9999.0)
    rf_args = (cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"])
    for method in ("time", "freq"):
        for rft in ("P", "S"):
            res[f"librf/fwd_{method}_{rft}"] = ctx.rf_forward(thk, rho, vp, vs, q, q, *rf_args, method, 0.001, rft)
        rf, drf = ctx.rf_kernel_all(thk, rho, vp, vs, q, q, *rf_args, method, 0.001, "P")
        res[f"librf/all_{method}_rf"], res[f"librf/all_{method}_drf"] = rf, drf
    np.savez(out, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="*")
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--worker", default=None)
    a = ap.parse_args()
    if a.worker:
        worker(a.worker, a.batch)
        return
    outs = []
    tmp = tempfile.mkdtemp()
    for i, lib in enumerate(a.libs):
        out = os.path.join(tmp, f"o{i}.npz")
        env = dict(os.environ, RFS_LIB="" if lib == "default" else os.path.abspath(lib))
        subprocess.run([sys.executable, __file__, "--worker", out, "--batch", str(a.batch)], env=env, check=True)
        outs.append(np.load(out))
    ref = outs[0]
    legs = sorted({k.split("/")[0] for k in ref.files})
    rc = 0
    for lib, o in zip(a.libs[1:], outs[1:]):
        for leg in legs:
            nbad = 0
            for k in (k for k in ref.files if k.split("/")[0] == leg):
                x, y = ref[k], o[k]
                same = (x.view(np.uint8) == y.view(np.uint8)).all() if x.dtype != object else True
                if not same:
                    neq = np.sum(~((x == y) | (np.isnan(x) & np.isnan(y)))) if x.dtype.kind == "f" else np.sum(x != y)
                    if neq:
                        nbad += 1
                        scale = np.nanmax(np.abs(x), axis=-1, keepdims=True) + 1e-300 if x.ndim > 1 else np.abs(x) + 1e-300
                        print(f"  {k}: {neq} of {x.size} values differ; max |diff| / max|row| "
                              f"{np.nanmax(np.abs(x - y) / scale):.3e}")
            print(f"{a.libs[0]} vs {lib} [{leg}]: {'BIT-IDENTICAL' if nbad == 0 else str(nbad) + ' arrays differ'}")
            rc |= nbad != 0
    sys.exit(rc)


if __name__ == "__main__":
    main()
