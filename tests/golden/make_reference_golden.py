"""Golden vectors from the REFERENCE'S OWN Python code:

    RFSURFHMC_REFERENCE=<checkout of the original RfSurfHmc> python tests/golden/make_reference_golden.py
                                                        ->  tests/golden/reference_code.npz

What runs unmodified from that checkout (imported, never copied):
  * model/model_surf.py, model/model_rf.py, model/model_rf_swd_vs_thk.py  -- Brocher relations,
    chain rule, residual contraction, joint weighting, failure convention   (SURVEY rows a1-a3)
  * pyhmc/hmc.py  (HamitonianMC)  and  pyhmc/hmcda.py  (HMCDualAveraging)  -- initial model,
    leapfrog, reflections, Metropolis, dual averaging, _find_initial_dt, NumPy's legacy global
    RNG stream                                                             (SURVEY rows a13, a14)
  * src/SWD/main.cpp, src/SWD/surfdisp.cpp, src/RF/main.cpp -- the pybind11 modules `libsurf` and
    `librf` themselves (float32 casts, retry loop, _RayleighGroup/_LoveGroup, _SurfKernel,
    _flat2sphere), compiled in place by `make -C oracle ref` into oracle/_ref/    (rows a5, a10, b)
What is stubbed, because it cannot exist here (gfortran / FFTW3 / h5py absent):
  * the Fortran entry points those modules call (surfdisp96_, sregn96_, slegn96_, sregnpu_,
    slegnpu_, cal_rf_*_) -> oracle/ref_fortran_shims.cpp forwards them to the C++ restatements of
    oracle/, which therefore stay the unpinned part;
  * `h5py` -> an in-memory stand-in (the samplers only write results through it).
The fixture pins oracle.surf_* / rf_* (the restated C++ layers), oracle.joint_batch (the restated
glue) and oracle/hmc_ref.py (the restated samplers) against the reference's real code on top of
the same numerics; tests never need the checkout.
"""
import contextlib
import io
import os
import sys
import types
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("RFSURFHMC_REFERENCE")     # a checkout of the original RfSurfHmc project
if not REF:
    sys.exit("set RFSURFHMC_REFERENCE to a checkout of the original RfSurfHmc project")
sys.path.insert(0, ROOT)
from oracle.oracle import Oracle  # noqa: E402

O = Oracle()


# ---------------------------------------------------------------- stubs
class _FakeH5File(dict):
    def __init__(self, *a, **k):
        super().__init__()

    def create_group(self, name):
        return None

    def create_dataset(self, name, data=None, dtype=None, shape=None):
        self[name] = np.array(data, dtype="f8") if data is not None else np.zeros(shape)
        return self[name]

    def close(self):
        pass


h5 = types.ModuleType("h5py")
h5.File = _FakeH5File
sys.modules["h5py"] = h5

import subprocess  # noqa: E402
subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + os.path.abspath(REF)],
                      stdout=subprocess.DEVNULL)
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
import libsurf  # noqa: E402  (the reference's own pybind11 module, built from its checkout)
import librf  # noqa: E402
lib = types.ModuleType("model.lib")
lib.__path__ = []
lib.libsurf, lib.librf = libsurf, librf
sys.path.insert(0, REF)
import model  # noqa: E402  (the reference's package)
sys.modules["model.lib"] = lib
sys.modules["model.lib.libsurf"] = libsurf
sys.modules["model.lib.librf"] = librf
model.lib = lib
from model.model_rf import ReceiverFunc  # noqa: E402
from model.model_surf import SurfWD  # noqa: E402
from model.model_rf_swd_vs_thk import Joint_RF_SWD  # noqa: E402
from pyhmc.hmc import HamitonianMC  # noqa: E402
from pyhmc.hmcda import HMCDualAveraging  # noqa: E402
import yaml  # noqa: E402


def build_model(param):
    """main_base.py:23-58, verbatim in behaviour"""
    model_swd = SurfWD.init(**param["swd"])
    model_rf = ReceiverFunc.init(**param["rf"])
    thk = np.asarray(param["true_model"]["thk"], dtype=float)
    vs = np.asarray(param["true_model"]["vs"], dtype=float)
    model_swd.set_thk(thk)
    model_rf.set_thk(thk)
    m = Joint_RF_SWD(1.0, 1.0, model_rf, model_swd)
    x = np.hstack((vs, thk))
    drsyn, dssyn, _ = m.forward(x)
    dobs = np.zeros(m.ndata)
    dobs[:m.rfmodel.nt] = drsyn
    dobs[m.rfmodel.nt:] = dssyn
    m.set_obsdata(dobs[:m.rfmodel.nt], dobs[m.rfmodel.nt:])
    n = len(x)
    b = np.ones((n, 2))
    for i in range(len(thk)):   # main_base.py:65-77
        b[i, 0] = max(vs[i] - vs[i] * 0.8, 1.5)
        b[i, 1] = min(vs[i] + vs[i] * 0.8, 5.0)
        b[i + len(thk), 0] = thk[i] - thk[i] * 0.2
        b[i + len(thk), 1] = thk[i] + thk[i] * 0.2
    b[-1, :] = 0.0, 2.0
    return m, x, dobs, b


def run_sampler(cls, m, b, rank, hparam, max_traj):
    """sample() of the reference class with its per-trajectory decisions recorded; the run is cut
    after max_traj trajectories by raising from the instrumented _leapfrog."""
    chain = cls.init(m, b, rank, **hparam)
    rec = {"accepts": [], "L": [], "dt": [], "x_after": []}
    orig = chain._leapfrog

    class _Stop(Exception):
        pass

    if cls is HamitonianMC:
        def wrapped(x, dt, L):
            if len(rec["accepts"]) >= max_traj:
                raise _Stop()
            out = orig(x, dt, L)
            rec["accepts"].append(1 if out[3] else 0)
            rec["L"].append(L)
            rec["dt"].append(dt)
            rec["x_after"].append(np.array(out[0], dtype=float).copy())
            return out
    else:
        # dual averaging: _leapfrog returns alpha; the accept draw happens in sample()
        state = {"pending": None}
        orig_rand = np.random.rand

        def wrapped(x, dt, L):
            if len(rec["L"]) >= max_traj:
                raise _Stop()
            out = orig(x, dt, L)
            rec["L"].append(L)
            rec["dt"].append(dt)
            rec["x_after"].append(np.array(out[0], dtype=float).copy())
            rec.setdefault("alpha", []).append(float(out[3]))
            return out
    chain._leapfrog = wrapped
    with contextlib.redirect_stdout(io.StringIO()):
        try:
            chain.sample()
        except _Stop:
            pass
    init = np.array(chain.fio["initmodel"], dtype=float)
    return chain, rec, init


def run_driver(script, sampler_cls, nsamples, ndraws, workdir):
    """Run the reference's main_base.py / main_DA.py UNMODIFIED as __main__ (single MPI rank) on a
    copy of its param.yaml with a short chain; returns what it wrote plus the bounds it built."""
    import runpy

    class _Comm:
        def Get_rank(self): return 0
        def Get_size(self): return 1
        def bcast(self, x, root=0): return x
        def Gather(self, src, dst, root=0): dst[0, :] = src

    mpi = types.ModuleType("mpi4py")
    mpi.MPI = types.SimpleNamespace(COMM_WORLD=_Comm())
    sys.modules["mpi4py"] = mpi
    for name in ("matplotlib", "matplotlib.colors", "matplotlib.pyplot"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib.colors"].BoundaryNorm = object
    param = yaml.safe_load(open(os.path.join(REF, "param.yaml")))
    param["hmc"].update(nsamples=nsamples, ndraws=ndraws, OUTPUT_DIR=os.path.join(workdir, "results") + "/")
    if sampler_cls is HMCDualAveraging:
        param["hmc"]["dt"] = 0.02
    os.makedirs(workdir, exist_ok=True)
    yaml.safe_dump(param, open(os.path.join(workdir, "param.yaml"), "w"))
    seen = {}
    orig_init = sampler_cls.__dict__["init"].__func__

    def spy(cls, model_, boundaries, rank, **kw):
        seen["bounds"] = np.array(boundaries, dtype=float).copy()
        return orig_init(cls, model_, boundaries, rank, **kw)
    sampler_cls.init = classmethod(spy)
    cwd = os.getcwd()
    os.chdir(workdir)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            runpy.run_path(os.path.join(REF, script), run_name="__main__")
    finally:
        os.chdir(cwd)
        sampler_cls.init = classmethod(orig_init)
    res = os.path.join(workdir, "results")
    return dict(bounds=seen["bounds"], real_syn=np.load(os.path.join(res, "real_syn.npy")),
                misfit=np.load(os.path.join(res, "misfit.npy")), dt=float(param["hmc"]["dt"]))


def run_test_forward(workdir):
    """The reference's only test script, test_forward.py (time-domain RF, nt=500, and Rc/Rg of a
    second model), run UNMODIFIED; the three curves it plots are captured from a stand-in pyplot."""
    import runpy
    calls = []
    plt = types.ModuleType("matplotlib.pyplot")
    plt.plot = lambda x, y, *a, **k: calls.append((np.array(x, dtype=float), np.array(y, dtype=float)))
    for name in ("figure", "subplot", "title", "savefig", "show", "legend", "xlabel", "ylabel"):
        setattr(plt, name, lambda *a, **k: None)
    mpl = types.ModuleType("matplotlib")
    colors = types.ModuleType("matplotlib.colors")
    colors.BoundaryNorm = object
    saved = {k: sys.modules.get(k) for k in ("matplotlib", "matplotlib.colors", "matplotlib.pyplot")}
    sys.modules.update({"matplotlib": mpl, "matplotlib.colors": colors, "matplotlib.pyplot": plt})
    mpl.pyplot, mpl.colors = plt, colors
    os.makedirs(workdir, exist_ok=True)
    cwd = os.getcwd()
    os.chdir(workdir)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            runpy.run_path(os.path.join(REF, "test_forward.py"), run_name="__main__")
    finally:
        os.chdir(cwd)
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
    assert len(calls) == 3
    return calls


def main():
    param = yaml.safe_load(open(os.path.join(REF, "param.yaml")))
    param["hmc"]["OUTPUT_DIR"] = "/tmp/rfs_ref_golden/"
    os.makedirs(param["hmc"]["OUTPUT_DIR"], exist_ok=True)
    m, x0, dobs, b = build_model(param)
    out = {"x_true": x0, "dobs": dobs, "bounds": b}

    # ---- the compiled modules themselves: every wave type, mode, flat / spherical earth; RF both
    # methods, both types, all parameter kernels
    thk, vs = x0[7:], x0[:7]
    vp, rho = m.swdmodel.empirical_relation(vs)
    T = np.asarray(param["swd"]["tRc"], dtype=float)
    models = [(thk, vp, vs, rho)]
    rr = np.random.default_rng(7)
    for _ in range(3):
        v = vs * (1 + 0.08 * rr.uniform(-1, 1, 7))
        a, r = m.swdmodel.empirical_relation(v)
        models.append((thk * (1 + 0.15 * rr.uniform(-1, 1, 7)) * (thk > 0), a, v, r))
    out["cpp_models"] = np.array([np.vstack(mm) for mm in models])
    out["cpp_T"] = T
    for im, (h, a, v, r) in enumerate(models):
        for wt in ("Rc", "Rg", "Lc", "Lg"):
            for mode in (0, 1, 2):
                for sph in (False, True):
                    if im > 0 and (mode == 2 or sph):
                        continue
                    c, ok = libsurf.forward(h, a, v, r, T, wt, mode, sph)
                    k = libsurf.adjoint_kernel(h, a, v, r, T, wt, mode, sph)
                    key = f"cpp{im}_{wt}_{mode}_{int(sph)}"
                    out[key + "_fwd"] = np.asarray(c)
                    out[key + "_ok"] = np.array([bool(ok), bool(k[5])])
                    for nm, arr in zip(("c", "da", "db", "dr", "dh"), k[:5]):
                        if wt[0] == "L" and nm == "da":
                            continue  # uninitialised memory in the reference (src/SWD/main.cpp:68)
                        out[key + "_k" + nm] = np.asarray(arr)
    q = thk * 0 + 9999.0
    rfa = (0.045, 125, 0.4, 1.5, 5.0)
    for method in ("freq", "time"):
        for rft in ("P", "S"):
            key = f"cpprf_{method}_{rft}"
            out[key + "_fwd"] = np.asarray(librf.forward(thk, rho, vp, vs, q, q, *rfa, method, 0.001, rft))
            d, kl = librf.kernel_all(thk, rho, vp, vs, q, q, *rfa, method, 0.001, rft)
            out[key + "_all"] = np.asarray(kl)
            for par in ("vs", "vp", "rho", "thick"):
                out[key + "_k" + par] = np.asarray(librf.kernel(thk, rho, vp, vs, q, q, *rfa, method, 0.001, rft, par)[1])

    # ---- glue: Joint / RF-only / SWD-only misfit_and_grad at a handful of models
    rng = np.random.default_rng(20240917)
    X = np.vstack((x0 * 1.02, x0 * (1 + 0.05 * rng.uniform(-1, 1, (6, x0.size))),
                   b[:, 0] + (b[:, 1] - b[:, 0]) * np.sort(rng.random((3, x0.size)), axis=1)))
    X[:, -1] = rng.uniform(0, 2, X.shape[0])
    U, G, D, F = [], [], [], []
    Ur, Gr, Us, Gs = [], [], [], []
    for x in X:
        u, g, d, f = m.misfit_and_grad(x)
        U.append(u); G.append(g); D.append(d); F.append(bool(f))
        ur, gr, _ = m.rfmodel.misfit_and_grad(x)
        us, gs, _, _ = m.swdmodel.misfit_and_grad(x)
        Ur.append(ur); Gr.append(gr); Us.append(us); Gs.append(gs)
    out.update(glue_X=X, glue_U=np.array(U), glue_grad=np.array(G), glue_dsyn=np.array(D),
               glue_flag=np.array(F), glue_U_rf=np.array(Ur), glue_grad_rf=np.array(Gr),
               glue_U_swd=np.array(Us), glue_grad_swd=np.array(Gs))

    # ---- samplers on the real joint model (short runs: the point is the decision sequence)
    hp = dict(param["hmc"], nsamples=40, ndraws=5)
    for rank in (0, 3):
        chain, rec, init = run_sampler(HamitonianMC, m, b, rank, hp, max_traj=14)
        out[f"base{rank}_init"] = init
        out[f"base{rank}_accepts"] = np.array(rec["accepts"])
        out[f"base{rank}_L"] = np.array(rec["L"])
        out[f"base{rank}_x"] = np.array(rec["x_after"])
    hp = dict(param["hmc"], nsamples=20, ndraws=4, dt=0.02)
    for rank in (0, 5):
        chain, rec, init = run_sampler(HMCDualAveraging, m, b, rank, hp, max_traj=8)
        out[f"da{rank}_init"] = init
        out[f"da{rank}_L"] = np.array(rec["L"])
        out[f"da{rank}_dt"] = np.array(rec["dt"])
        out[f"da{rank}_alpha"] = np.array(rec["alpha"])
        out[f"da{rank}_x"] = np.array(rec["x_after"])
    # ---- test_forward.py, the reference's own (and only) test script
    (t_rf, rf), (tRc, rc), (tRg, rg) = run_test_forward("/tmp/rfs_ref_golden/test_forward")
    out.update(tf_t=t_rf, tf_rf=rf, tf_tRc=tRc, tf_Rc=rc, tf_tRg=tRg, tf_Rg=rg)

    # ---- the drivers themselves, end to end (main_base.py / main_DA.py as __main__, one rank)
    for tag, script, cls, ns, ndr in (("drvbase", "main_base.py", HamitonianMC, 10, 3),
                                      ("drvda", "main_DA.py", HMCDualAveraging, 6, 3)):
        r = run_driver(script, cls, ns, ndr, f"/tmp/rfs_ref_golden/{tag}")
        out[tag + "_bounds"], out[tag + "_real_syn"], out[tag + "_misfit"] = r["bounds"], r["real_syn"], r["misfit"]
        out[tag + "_cfg"] = np.array([ns, ndr, r["dt"]], dtype=float)
    out["base_hparam"] = np.array([0.1, 5, 20, 991206, 40, 5], dtype=float)
    out["da_hparam"] = np.array([0.02, 10, 0.65, 991206, 20, 4], dtype=float)
    np.savez_compressed(os.path.join(HERE, "reference_code.npz"), **out)
    print("wrote reference_code.npz:", {k: np.shape(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
