"""Golden vectors for rfsurfhmc_b200/utils.py from the reference's own src/utils.py, imported
unmodified from a checkout of the original RfSurfHmc project (matplotlib, which that module imports but
the two functions do not use, is replaced by an empty stand-in when absent):
    RFSURFHMC_REFERENCE=<checkout> python tests/golden/make_utils_golden.py   -> tests/golden/utils_resample.npz"""
import importlib.util
import os
import sys
import types
import numpy as np

try:
    import matplotlib.pyplot  # noqa: F401
except Exception:
    m = types.ModuleType("matplotlib")
    m.pyplot = types.ModuleType("matplotlib.pyplot")
    sys.modules["matplotlib"] = m
    sys.modules["matplotlib.pyplot"] = m.pyplot
REF = os.environ.get("RFSURFHMC_REFERENCE")     # a checkout of the original RfSurfHmc project
if not REF:
    sys.exit("set RFSURFHMC_REFERENCE to a checkout of the original RfSurfHmc project")
spec = importlib.util.spec_from_file_location("ref_utils", os.path.join(REF, "src", "utils.py"))
ref = importlib.util.module_from_spec(spec)
spec.loader.exec_module(ref)

rng = np.random.default_rng(42)
out = {}
cases = [(0.1, -10.0, 60.0, -5.0, 30.0), (0.025, -5.0, 40.0, -2.0, 20.5), (0.4, -20.0, 120.0, -5.0, 45.0)]
for i, (dt, t0, t1, ts, te) in enumerate(cases):
    t = np.arange(t0, t1, dt)
    d = np.exp(-0.5 * ((t - 0.0) / 0.8)**2) + 0.3 * np.exp(-0.5 * ((t - 4.2) / 1.0)**2) + 0.02 * rng.standard_normal(t.size)
    y, nt, dtn, shift = ref.get_rf_inv_para(d, t, ts, te)
    out[f"in_{i}_t"], out[f"in_{i}_d"] = t, d
    out[f"in_{i}_win"] = np.array([ts, te])
    out[f"out_{i}_y"] = y
    out[f"out_{i}_meta"] = np.array([nt, dtn, shift])
out["pow2_in"] = np.array([0, 1, 2, 3, 5, 64, 65, 1000, 4096, 4097])
out["pow2_out"] = np.array([ref.next_power_of_2(int(v)) for v in out["pow2_in"]])
np.savez(os.path.join(os.path.dirname(os.path.abspath(__file__)), "utils_resample.npz"), **out)
print("written", len(cases), "cases")
