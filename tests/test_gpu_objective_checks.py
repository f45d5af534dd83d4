"""The three evaluations of the objective (rfs_misfit_grad_sets_dev, rfs_misfit_grad_sets_host and
rfs_hmc_run_sets) check their arguments and the context's configuration with one rule set: an input
that breaks exactly one rule gets the same code from each of them."""
import numpy as np
import pytest
import torch
from rfsurfhmc_b200._lib import Context, RfsError
from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds

pytestmark = pytest.mark.gpu
RFS_E_ARG, RFS_E_CONFIG = -2, -4
N, ROWS = 7, 4
ENTRIES = ("dev", "host", "hmc")
NAMES = {"dev": "rfs_misfit_grad_sets_dev", "host": "rfs_misfit_grad_sets_host", "hmc": "rfs_hmc_run_sets"}


def _context(swd=True, rf=True, obs=True, S=1, rf_layers=N, extra=0):
    """F1 context with the given parts configured; dobs [S][ndata + extra]."""
    cfg = f1_config()
    c = Context(0)
    if swd:
        c.config_swd(N, tRc=cfg["tRc"], tRg=cfg["tRg"])
    if rf:
        c.config_rf(rf_layers, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                    cfg["rf_type"], cfg["method"])
    if obs:
        d = np.zeros((S, c.ndata(0) + extra))
        c.config_obs(d[0] if S == 1 else d)
    return c


def _call(c, entry, which, sets):
    x = np.tile(f1_true_model(), (ROWS, 1))
    if entry == "host":
        c.misfit_grad_host(x, which, sets=sets)
    elif entry == "dev":
        dev = torch.device("cuda", 0)
        xd = torch.from_numpy(x).to(dev)
        U = torch.zeros(ROWS, dtype=torch.float64, device=dev)
        G = torch.zeros_like(xd)
        D = torch.zeros((ROWS, max(c.ndata(which), 1)), dtype=torch.float64, device=dev)
        F = torch.zeros(ROWS, dtype=torch.uint8, device=dev)
        sd = None if sets is None else torch.tensor(sets, dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream(dev)
        c.misfit_grad_dev(ROWS, xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                          st.cuda_stream, sets_ptr=0 if sd is None else sd.data_ptr())
        st.synchronize()
    else:
        c.hmc_run(0, np.arange(ROWS), driver_bounds(f1_true_model()), 0.1, nsamples=2, ndraws=1, max_iters=2,
                  which=which, sets=sets)


def _code(c, entry, which, sets=None):
    try:
        _call(c, entry, which, sets)
    except RfsError as e:
        return e.code, str(e)
    return 0, ""


# (name, context, which, with a set array, expected code)
SINGLE_FAULTS = [
    ("which_negative", {}, -1, False, RFS_E_ARG),
    ("which_too_large", {}, 3, True, RFS_E_ARG),
    ("no_swd_joint", dict(swd=False), 0, False, RFS_E_CONFIG),
    ("no_swd_swd_only", dict(swd=False), 2, True, RFS_E_CONFIG),
    ("no_rf_joint", dict(rf=False), 0, True, RFS_E_CONFIG),
    ("no_rf_rf_only", dict(rf=False), 1, False, RFS_E_CONFIG),
    ("no_obs", dict(obs=False), 0, False, RFS_E_CONFIG),
    ("no_set_array", dict(S=3), 0, False, RFS_E_CONFIG),
    ("layer_counts_differ", dict(rf_layers=N - 1), 0, False, RFS_E_CONFIG),
    ("dobs_too_long", dict(extra=1), 0, True, RFS_E_CONFIG),
    ("dobs_too_short", dict(extra=-1), 0, False, RFS_E_CONFIG),
]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("name,kw,which,with_sets,code", SINGLE_FAULTS, ids=[f[0] for f in SINGLE_FAULTS])
def test_single_fault_code(entry, name, kw, which, with_sets, code):
    c = _context(**kw)
    try:
        got, msg = _code(c, entry, which, [0] * ROWS if with_sets else None)
        assert got == code, msg
        if name == "no_set_array":
            assert NAMES[entry] in msg, msg
    finally:
        c.close()


@pytest.mark.parametrize("entry", ENTRIES)
def test_configured_context_passes_the_check(entry):
    c = _context(S=2)
    try:
        assert _code(c, entry, 0, [0, 1, 1, 0]) == (0, "")
    finally:
        c.close()


@pytest.mark.parametrize("entry", ENTRIES)
def test_set_array_without_observations_is_a_configuration_error(entry):
    """A set array on a context that holds no observations is RFS_E_CONFIG from every entry point.
    rfs_misfit_grad_sets_host used to report RFS_E_ARG here (each index outside [0, 0))."""
    c = _context(obs=False)
    try:
        assert _code(c, entry, 0, [0] * ROWS)[0] == RFS_E_CONFIG
    finally:
        c.close()
