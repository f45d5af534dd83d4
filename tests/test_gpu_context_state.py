"""A context carries one configured fused objective and also serves the libsurf / librf drop-ins. A
drop-in call with its own receiver-function settings must leave that objective as it was: the next
fused evaluation on the context returns the same bits as the one before it."""
import numpy as np
import pytest
from oracle.oracle import brocher
from rfsurfhmc_b200._lib import Context
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, perturbed_models

pytestmark = pytest.mark.gpu


def _dropins(c, x):
    """Drop-in calls on the models x. The RF calls use the F2 "smoke-time" sampling of the reference's
    test_forward.py (nt = 500, dt = 0.1: a 512-point transform, where F1 has 128 points)."""
    n = x.shape[1] // 2
    vs, thk = x[:, :n], x[:, n:]
    vp, rho = brocher(vs)
    q = np.full_like(thk, 9999.)
    f2 = (thk, rho, vp, vs, q, q, 0.045, 500, 0.1, 1.0, 5.0)
    out = {}
    for method in ("freq", "time"):
        out["rf_forward_" + method] = c.rf_forward(*f2, method=method)
    out["rf_kernel_all_rf"], out["rf_kernel_all_drf"] = c.rf_kernel_all(*f2, method="freq")
    for name, a in zip(("c", "dcda", "dcdb", "dcdr", "dcdh", "ok"),
                       c.surf_adjoint_kernel(thk, vp, vs, rho, f1_config()["tRc"], "Rg")):
        out["surf_adjoint_kernel_" + name] = a
    return out


def test_dropins_leave_the_fused_objective_unchanged(ctx):
    cfg = f1_config()
    x0 = f1_true_model()
    n = x0.size // 2
    rays = [0.045, 0.06]
    ctx.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
    ctx.config_rf(n, rays, cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                  cfg["rf_type"], cfg["method"])
    ctx.config_obs(np.zeros(ctx.ndata()))
    _, _, d0, _ = ctx.misfit_grad_host(x0[None, :])
    ctx.config_obs(d0[0])
    X = perturbed_models(x0, 64, seed=21, rel=0.1)

    first = ctx.misfit_grad_host(X)
    got = _dropins(ctx, X[:8])
    second = ctx.misfit_grad_host(X)
    for name, a, b in zip(("U", "grad", "dsyn", "flag"), first, second):
        assert np.array_equal(a, b), name

    fresh = Context(0)
    try:
        want = _dropins(fresh, X[:8])
    finally:
        fresh.close()
    for key in want:
        assert np.array_equal(got[key], want[key]), key
