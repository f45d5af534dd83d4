"""Receiver functions at several Gaussian widths in one objective (rfs_config_rf_gauss) against the same
widths as one-width contexts evaluated in turn.

    python tools/rf_gauss_bench.py [--reps 5] [--out profiles/rf_gauss_bench.json]

  (a) RF only, frequency method, n = 40, nt = 2048, dt = 0.05, rays 0.04/0.06/0.08, 16 384 models:
      G = 1, 2, 3 widths (1.0, 2.5, 5.0) in one context, against G one-width contexts evaluated in
      turn, plus the per-kernel times of one G = 1 and one G = 2 evaluation (rfs_profile_eval);
  (b) F1 joint (the reference's param.yaml), 16 384 chain states: widths [1.5] against [1.5, 2.5] (the RF
      branch runs beside the root search);
  (c) RF only, time method, F1 layers and sampling, 1 024 models: one width against two;
  (d) base-sampler HMC, 1 024 chains, F1 joint objective with widths [1.5, 2.5] (and [1.5] for scale):
      evaluations per second over a fixed number of trajectories.
In (a)-(c) the variants alternate within each repetition; each timing is a host clock around work that
ends in a device synchronise, after every shape was warmed up.  Median, min and max over --reps
repetitions.  Prints one JSON line and writes it to --out with the card name, power limit and max SM
clock read in the same run."""
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


def spread(ts):
    ts = np.asarray(ts) * 1e3
    return {"median_ms": float(np.median(ts)), "min_ms": float(ts.min()), "max_ms": float(ts.max()),
            "reps": int(ts.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--models", type=int, default=16384)
    ap.add_argument("--hmc-iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rf_gauss_bench.json"))
    a = ap.parse_args()
    import torch
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models
    from bench import layered_models
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    cfg, x0 = f1_config(), f1_true_model()
    res = {**gpu_info(), "reps": a.reps}

    def context(which, n, rays, nt, dt, gauss, method, dobs):
        c = Context(0)
        if which != 1:
            c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
        c.config_rf(n, rays, nt, dt, gauss, cfg["time_shift"], cfg["water"], "P", method)
        c.config_obs(dobs)
        return c

    def buffers(c, which, Xd):
        B = Xd.shape[0]
        return (torch.empty(B, dtype=torch.float64, device=dev), torch.empty(Xd.shape, dtype=torch.float64, device=dev),
                torch.empty(B, c.ndata(which), dtype=torch.float64, device=dev),
                torch.empty(B, dtype=torch.uint8, device=dev))

    def evaluator(cs, which, Xd):
        """one call: every context of cs evaluated in turn on Xd"""
        bufs = [buffers(c, which, Xd) for c in cs]

        def run():
            for c, (U, G, D, F) in zip(cs, bufs):
                c.misfit_grad_dev(Xd.shape[0], Xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(),
                                  F.data_ptr(), st.cuda_stream)
        return run

    def alternate(variants, inner=1):
        """variants: {name: run}; warmed up, then timed in turn within each repetition"""
        for fn in variants.values():
            fn()
        torch.cuda.synchronize()
        ts = {k: [] for k in variants}
        for _ in range(a.reps):
            for k, fn in variants.items():
                t0 = time.perf_counter()
                for _ in range(inner):
                    fn()
                torch.cuda.synchronize()
                ts[k].append((time.perf_counter() - t0) / inner)
        return {k: spread(v) for k, v in ts.items()}

    def close(cs):
        for c in cs:
            c.close()

    # (a) RF only, frequency method, C3 sizes
    n, nt, dt = 40, 2048, 0.05
    rays, widths = [0.04, 0.06, 0.08], [1.0, 2.5, 5.0]
    Xd = torch.from_numpy(layered_models(a.models, n, 2)).to(dev)
    dobs = 0.01 * np.random.default_rng(3).standard_normal(3 * 3 * nt)
    # five contexts side by side: a 24 GB workspace budget each runs the batch in one chunk (22 GB of
    # derivative spectra) and keeps them all on the card together
    old = os.environ.get("RFS_WS_BUDGET_MB")
    os.environ["RFS_WS_BUDGET_MB"] = "24000"
    try:
        one = [context(1, n, rays, nt, dt, w, "freq", dobs[:3 * nt]) for w in widths]
        multi = {G: context(1, n, rays, nt, dt, widths[:G], "freq", dobs[:3 * G * nt]) for G in (2, 3)}
    finally:
        if old is None:
            del os.environ["RFS_WS_BUDGET_MB"]
        else:
            os.environ["RFS_WS_BUDGET_MB"] = old
    variants = {"G1": evaluator(one[:1], 1, Xd)}
    for G in (2, 3):
        variants[f"G{G}_one_context"] = evaluator([multi[G]], 1, Xd)
        variants[f"G{G}_one_width_contexts"] = evaluator(one[:G], 1, Xd)
    t = alternate(variants)
    leg = {"workload": "RF only (freq), n=40, nt=2048, dt=0.05, rays 0.04/0.06/0.08, widths 1.0/2.5/5.0, "
                       "%d models" % a.models, "times": t}
    for G in (2, 3):
        leg[f"G{G}_one_context_over_one_width_contexts"] = (t[f"G{G}_one_context"]["median_ms"] /
                                                           t[f"G{G}_one_width_contexts"]["median_ms"])
        leg[f"G{G}_one_context_over_G1"] = t[f"G{G}_one_context"]["median_ms"] / t["G1"]["median_ms"]
    prof = {}
    for name, c, which in (("G1", one[0], 1), ("G2", multi[2], 1)):
        U, G_, D, F = buffers(c, which, Xd)
        p = c.profile_eval(Xd.shape[0], Xd.data_ptr(), which, U.data_ptr(), G_.data_ptr(), D.data_ptr(),
                           F.data_ptr(), st.cuda_stream)
        prof[name] = {k: {"ms": v[0], "launches": v[1]} for k, v in p.items() if v[1] > 0}
    leg["kernels_one_evaluation"] = prof
    res["a_rf_freq_c3"] = leg
    close(one + list(multi.values()))
    print(json.dumps({"a": leg}), file=sys.stderr, flush=True)
    del Xd
    torch.cuda.empty_cache()

    # (b) F1 joint, 16 384 chain states
    n = x0.size // 2
    X = np.vstack((perturbed_models(x0, a.models // 2, 11, rel=0.1),
                   perturbed_models(x0, a.models - a.models // 2, 12, rel=0.3)))
    Xd = torch.from_numpy(X).to(dev)
    d1 = 0.01 * np.random.default_rng(5).standard_normal(cfg["nt"] * 2 + 72)
    cs = {"G1": context(0, n, cfg["ray_p"], cfg["nt"], cfg["dt"], [1.5], "freq",
                        np.concatenate((d1[:cfg["nt"]], d1[2 * cfg["nt"]:]))),
          "G2": context(0, n, cfg["ray_p"], cfg["nt"], cfg["dt"], [1.5, 2.5], "freq", d1)}
    t = alternate({k: evaluator([c], 0, Xd) for k, c in cs.items()}, inner=10)
    res["b_f1_joint"] = {"workload": "F1 joint, %d chain states, widths [1.5] vs [1.5, 2.5]" % a.models, "times": t,
                         "G2_over_G1": t["G2"]["median_ms"] / t["G1"]["median_ms"]}
    close(cs.values())
    print(json.dumps({"b": res["b_f1_joint"]}), file=sys.stderr, flush=True)

    # (c) time method, F1 sizes, 1 024 models
    Xt = Xd[:1024].contiguous()
    d1 = 0.01 * np.random.default_rng(6).standard_normal(2 * cfg["nt"])
    cs = {"G1": context(1, n, cfg["ray_p"], cfg["nt"], cfg["dt"], [1.5], "time", d1[:cfg["nt"]]),
          "G2": context(1, n, cfg["ray_p"], cfg["nt"], cfg["dt"], [1.5, 2.5], "time", d1)}
    t = alternate({k: evaluator([c], 1, Xt) for k, c in cs.items()}, inner=5)
    res["c_rf_time_f1"] = {"workload": "RF only (time), F1 layers and sampling, 1024 models, widths [1.5] vs "
                                       "[1.5, 2.5]", "times": t, "G2_over_G1": t["G2"]["median_ms"] / t["G1"]["median_ms"]}
    close(cs.values())
    print(json.dumps({"c": res["c_rf_time_f1"]}), file=sys.stderr, flush=True)

    # (d) base-sampler HMC, 1 024 chains
    bounds = driver_bounds(x0)
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    hmc = {"workload": "base sampler, 1024 chains, F1 joint, %d trajectories per chain" % a.hmc_iters}
    for name, w in (("G1", [1.5]), ("G2", [1.5, 2.5])):
        c = Context(0)
        c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
        c.config_rf(n, cfg["ray_p"], cfg["nt"], cfg["dt"], w, cfg["time_shift"], cfg["water"], "P", "freq")
        c.config_obs(np.zeros(c.ndata(0)))
        _, _, d, _ = c.misfit_grad_host(x0[None, :], 0)
        c.config_obs(d[0])
        c.hmc_run(0, np.arange(1024), bounds, **kw)
        ts, evs = [], 0
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            evs = c.hmc_run(0, np.arange(1024), bounds, **kw)["evals"]
            ts.append(time.perf_counter() - t0)
        hmc[name] = {**spread(ts), "evals": int(evs), "evals_per_s": float(evs / np.median(ts))}
        c.close()
    res["d_hmc"] = hmc
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
