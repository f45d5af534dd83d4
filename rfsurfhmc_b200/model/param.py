"""Model-vector layout shared by the three objectives.

x = [vs(n), thk(n)] (the reference's parameterisation, vp and rho from Brocher's polynomials of vs), or
with vpvs=True x = [vs(n), thk(n), k(n)], k the Vp/Vs ratio of each layer: vp = k vs and rho = Brocher's
density polynomial of that vp (include/rfsurfhmc.h: rfs_config_param)."""
import numpy as np


def npar(vpvs):
    """Parameter blocks per layer: 3 with Vp/Vs, 2 without."""
    return 3 if vpvs else 2


def layer_count(width, vpvs):
    """Layer count n of a model vector of `width` columns; ValueError unless width = P n with n >= 2."""
    P = npar(vpvs)
    if width % P or width < 2 * P:
        layout = "[vs, thk, vpvs]" if vpvs else "[vs, thk]"
        raise ValueError(f"model vectors of {width} values do not hold {layout} blocks of n >= 2 layers "
                         f"({P} n values)")
    return width // P


def split(x, vpvs):
    """(vs, thk, k) of one model vector; k is None without Vp/Vs."""
    x = np.asarray(x, dtype=np.float64)
    n = layer_count(x.shape[-1], vpvs)
    return x[..., :n], x[..., n:2 * n], (x[..., 2 * n:] if vpvs else None)


def brocher(vs, k=None, deriv=False):
    """vp, rho (and drho/dvp, dvp/dvs when deriv): Brocher's polynomials, or vp = k vs when k is given."""
    if k is None:
        vp = 0.9409 + 2.0947 * vs - 0.8206 * vs**2 + 0.2683 * vs**3 - 0.0251 * vs**4
        dadb = 2.0947 - 0.8206 * 2 * vs + 0.2683 * 3 * vs**2 - 0.0251 * 4 * vs**3
    else:
        vp = k * vs
        dadb = k * 1.0
    rho = 1.6612 * vp - 0.4721 * vp**2 + 0.0671 * vp**3 - 0.0043 * vp**4 + 0.000106 * vp**5
    if not deriv:
        return vp, rho
    drda = 1.6612 - 0.4721 * 2 * vp + 0.0671 * 3 * vp**2 - 0.0043 * 4 * vp**3 + 0.000106 * 5 * vp**4
    return vp, rho, drda, dadb


def check_vpvs_box(bounds, vpvs):
    """bounds [..., P n, 2]: the Vp/Vs block's lower bounds must be > 1 (vp > vs)."""
    if not vpvs:
        return
    b = np.asarray(bounds, dtype=np.float64)
    n = layer_count(b.shape[-2], True)
    lo = b[..., 2 * n:, 0]
    if not np.all(lo > 1.0):
        raise ValueError(f"Vp/Vs bounds must have lower bounds > 1, got min {float(np.min(lo))}")
