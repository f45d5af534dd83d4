"""Cost of the [vs, thk, vpvs] parameterisation (rfs_config_param RFS_PARAM_VS_THK_VPVS) against the
default Brocher [vs, thk] one, on the same models (k = Brocher vp / vs), the two contexts alternating:

  f1   F1 joint objective (the flagship step), --chains rows in one evaluation
  c3   RF-only objective, frequency method, n = 40, nt = 2048, three ray parameters (BASELINE C3-like)
  hmc  base-sampler HMC, F1 joint, --hmc-chains chains x --hmc-iters trajectories: evaluations per second

Each figure is the median and min-max of --reps timed calls (device synchronised), written as one JSON
line to --out together with the card name and power limit read in the same run.

    python tools/vpvs_bench.py [--reps 5] [--out profiles/vpvs_bench.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def spread(ts, scale=1e3):
    ts = np.asarray(ts) * scale
    return {"median": float(np.median(ts)), "min": float(ts.min()), "max": float(ts.max()), "reps": int(ts.size)}


def with_k(X2):
    from oracle.oracle import brocher
    n = X2.shape[1] // 2
    vs = X2[:, :n]
    return np.hstack((X2, brocher(vs)[0] / vs))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--chains", type=int, default=16384)
    ap.add_argument("--c3-rows", type=int, default=2048)
    ap.add_argument("--hmc-chains", type=int, default=1024)
    ap.add_argument("--hmc-iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "vpvs_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vpvs_bench.py measures on a CUDA device; none is available")
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import (f1_config, f1_true_model, driver_bounds, driver_bounds_vpvs,
                                         perturbed_models)
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    res = {"tool": "vpvs_bench", **gpu_info(), "reps": a.reps}

    def contexts(setup):
        cs = {}
        for name, vpvs in (("brocher", False), ("vpvs", True)):
            c = Context(0)
            c.config_param(vpvs)
            setup(c)
            cs[name] = c
        return cs

    def alternate(cs, X2, which):
        """time one evaluation of every row in each context, alternating; returns ms statistics"""
        Xs = {"brocher": torch.from_numpy(X2).to(dev), "vpvs": torch.from_numpy(with_k(X2)).to(dev)}
        B = X2.shape[0]
        nd = cs["brocher"].ndata(which)
        out = {k: (torch.empty(B, dtype=torch.float64, device=dev),
                   torch.empty(B, Xs[k].shape[1], dtype=torch.float64, device=dev),
                   torch.empty(B, nd, dtype=torch.float64, device=dev),
                   torch.empty(B, dtype=torch.uint8, device=dev)) for k in cs}

        def call(k):
            U, G, D, F = out[k]
            cs[k].misfit_grad_dev(B, Xs[k].data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(),
                                  F.data_ptr(), st.cuda_stream)
        ts = {k: [] for k in cs}
        for k in cs:  # warm-up: module load, workspace growth
            call(k)
            call(k)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for k in cs:
                t0 = time.perf_counter()
                call(k)
                torch.cuda.synchronize()
                ts[k].append(time.perf_counter() - t0)
        r = {k: spread(v) for k, v in ts.items()}
        r["vpvs_over_brocher"] = r["vpvs"]["median"] / r["brocher"]["median"] - 1.0
        U2, U3 = out["brocher"][0].cpu().numpy(), out["vpvs"][0].cpu().numpy()
        ok = out["brocher"][3].cpu().numpy().astype(bool)
        r["max_rel_U_difference"] = float(np.max(np.abs(U3[ok] - U2[ok]) / np.maximum(np.abs(U2[ok]), 1e-300)))
        return r

    cfg, x0 = f1_config(), f1_true_model()
    n = x0.size // 2

    def f1_setup(c):
        c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
        c.config_rf(n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                    cfg["rf_type"], cfg["method"])
    cs = contexts(f1_setup)
    # observations: the Brocher synthetics of a perturbed truth
    cs["brocher"].config_obs(np.zeros(cs["brocher"].ndata()))
    dobs = cs["brocher"].misfit_grad_host(perturbed_models(x0, 1, seed=3, rel=0.03))[2][0]
    for c in cs.values():
        c.config_obs(dobs)
    X2 = perturbed_models(x0, a.chains, seed=11, rel=0.1)
    res["f1"] = {"rows": a.chains, "unit": "ms per evaluation", **alternate(cs, X2, 0)}

    # HMC, base sampler: the same chains in both parameterisations (k box +-10 % around Brocher's vp/vs)
    xk = with_k(x0[None, :])[0]
    boxes = {"brocher": driver_bounds(x0), "vpvs": driver_bounds_vpvs(xk)}
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    ids = np.arange(a.hmc_chains)
    hmc = {"chains": a.hmc_chains, "max_iters": a.hmc_iters, "unit": "s per run"}
    for k in cs:
        cs[k].hmc_run(0, ids[:64], boxes[k], **kw)
    ts = {k: [] for k in cs}
    evs = {}
    for _ in range(max(1, (a.reps + 1) // 2)):
        for k in cs:
            t0 = time.perf_counter()
            evs[k] = cs[k].hmc_run(0, ids, boxes[k], **kw)["evals"]
            ts[k].append(time.perf_counter() - t0)
    for k in cs:
        hmc[k] = {**spread(ts[k], 1.0), "evals": int(evs[k]), "evals_per_s": float(evs[k] / np.median(ts[k]))}
    res["hmc"] = hmc
    for c in cs.values():
        c.close()

    # C3-like RF only: n = 40, nt = 2048, three ray parameters
    n3 = 40
    rays = [0.04, 0.06, 0.08]
    i = np.arange(n3 - 1)
    vs = 2.0 + 2.7 * (np.arange(n3) / (n3 - 1))**0.7
    thk = np.hstack((0.5 + 0.1 * i, [0.0]))
    x3 = np.hstack((vs, thk))

    def c3_setup(c):
        c.config_rf(n3, rays, 2048, 0.05, 2.5, 5.0, 0.001, "P", "freq")
    cs = contexts(c3_setup)
    cs["brocher"].config_obs(np.zeros(3 * 2048))
    dobs = cs["brocher"].misfit_grad_host(x3[None, :] * 1.02, which=1)[2][0]
    for c in cs.values():
        c.config_obs(dobs)
    rng = np.random.default_rng(5)
    X2 = x3 * (1 + 0.03 * rng.uniform(-1, 1, (a.c3_rows, 2 * n3)))
    X2[:, -1] = 0.0
    res["c3"] = {"rows": a.c3_rows, "n": n3, "nt": 2048, "nray": 3, "unit": "ms per evaluation",
                 **alternate(cs, X2, 1)}
    for c in cs.values():
        c.close()

    line = json.dumps(res)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
