"""Named workloads shared by tests, smoke() and bench.py (SURVEY.md §8c/d).

F1 "default-freq" is the reference's own param.yaml (param.yaml:1-31); the bounds are the ones
main_base.py builds (main_base.py:65-77)."""
import numpy as np


def f1_true_model():
    vs = np.array([3.2, 2.8, 3.46, 3.3, 3.9, 4.5, 4.7])
    thk = np.array([6., 6., 13., 5., 10., 30., 0.])
    return np.hstack((vs, thk))


def f1_config():
    T = np.arange(5., 41.)
    return dict(tRc=T, tRg=T.copy(), tLc=[], tLg=[], mode=0, sphere=False, ray_p=0.045, nt=125, dt=0.4,
                gauss=1.5, time_shift=5., water=0.001, rf_type="P", method="freq", sigma1=1.0,
                sigma2=1.0, stale=True)


def driver_bounds(x_true):
    """main_base.py:65-77: vs +-80 % clipped to [1.5, 5], thk +-20 %, last thk in [0, 2]."""
    n = x_true.size // 2
    vs, thk = x_true[:n], x_true[n:]
    b = np.ones((2 * n, 2))
    b[:n, 0] = np.maximum(vs - vs * 0.8, 1.5)
    b[:n, 1] = np.minimum(vs + vs * 0.8, 5.0)
    b[n:, 0] = thk - thk * 0.2
    b[n:, 1] = thk + thk * 0.2
    b[-1, :] = 0.0, 2.0
    return b


def driver_bounds_vpvs(x_true):
    """Box of the [vs, thk, vpvs] parameterisation: driver_bounds for vs and thk, Vp/Vs +-10 % of the
    true value."""
    n = x_true.size // 3
    k = x_true[2 * n:]
    return np.vstack((driver_bounds(x_true[:2 * n]), np.stack((k * 0.9, k * 1.1), axis=1)))


def sorted_uniform_models_vpvs(bounds, B, seed):
    """sorted_uniform_models for [vs, thk, vpvs] boxes [3n, 2]: vs sorted ascending, thk and Vp/Vs
    permuted alike (the rule of the device HMC's initial models)."""
    rng = np.random.default_rng(seed)
    n = bounds.shape[0] // 3
    X = bounds[:, 0] + (bounds[:, 1] - bounds[:, 0]) * rng.random((B, 3 * n))
    idx = np.argsort(X[:, :n], axis=1)
    for j in range(3):
        X[:, j * n:(j + 1) * n] = np.take_along_axis(X[:, j * n:(j + 1) * n], idx, axis=1)
    return X


def sorted_uniform_models(bounds, B, seed):
    """Uniform draws in the box, vs sorted ascending with thk permuted alike — the distribution of
    HamitonianMC.set_initial_model (pyhmc/hmc.py:74-93), without the in-bounds redraw."""
    rng = np.random.default_rng(seed)
    n = bounds.shape[0] // 2
    X = bounds[:, 0] + (bounds[:, 1] - bounds[:, 0]) * rng.random((B, 2 * n))
    idx = np.argsort(X[:, :n], axis=1)
    X[:, :n] = np.take_along_axis(X[:, :n], idx, axis=1)
    X[:, n:] = np.take_along_axis(X[:, n:], idx, axis=1)
    return X


def perturbed_models(x_true, B, seed, rel=0.05):
    """Models near the truth (what chains look like after burn-in)."""
    rng = np.random.default_rng(seed)
    X = x_true * (1.0 + rel * rng.uniform(-1, 1, size=(B, x_true.size)))
    X[:, -1] = rng.uniform(0, 2, size=B)
    return X
