"""Station arrays on one GPU: one grouped evaluation over many stations vs one small batch per station.

    python tools/stations_bench.py [--reps 5] [--out profiles/stations_bench.json]

Forward configuration F1 (the reference's param.yaml), 16 384 models in total, split as (stations S,
models per station K) = (256, 64), (64, 256), (1024, 16):
  (a) grouped : one rfs_misfit_grad_sets_dev call over all S*K rows (row b on station b // K);
  (b) per-sta : what a user does without observation sets: for each station config_obs(dobs[s]) and one
                misfit_grad_dev of its K rows, one station after another, timed around the whole loop;
  (c) one set : the same 16 384 models against one observation vector (the cost of the set lookup).
HMC: 16 stations x 64 chains, base sampler, fixed max_iters: one hmc_run over all stations vs 16
sequential single-station runs.
Every shape is warmed up first; each timing is repeated --reps times (median, min, max reported), with a
host clock around work that ends in a device synchronise.  Station observations are the forward model
of seeded perturbations of the F1 true model plus seeded noise.  Prints one JSON line and writes it to
--out together with the card name and power limit read in the same run."""
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
    ap.add_argument("--total", type=int, default=16384)
    ap.add_argument("--hmc-iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stations_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stations_bench.py measures on a CUDA device; none is available")
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models

    cfg, x0 = f1_config(), f1_true_model()
    n = x0.size // 2
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    c = Context(0)
    c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
    c.config_rf(n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                cfg["rf_type"], cfg["method"])
    nd = c.ndata()

    def station_obs(S, seed):
        c.config_obs(np.zeros(nd))
        _, _, d, _ = c.misfit_grad_host(perturbed_models(x0, S, seed=seed, rel=0.05))
        return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)

    B = a.total
    X = torch.from_numpy(perturbed_models(x0, B, seed=11, rel=0.1)).to(dev)
    U = torch.empty(B, dtype=torch.float64, device=dev)
    G = torch.empty(B, 2 * n, dtype=torch.float64, device=dev)
    D = torch.empty(B, nd, dtype=torch.float64, device=dev)
    F = torch.empty(B, dtype=torch.uint8, device=dev)

    def call(off, rows, sets_ptr=0):
        c.misfit_grad_dev(rows, X[off].data_ptr(), 0, U[off].data_ptr(), G[off].data_ptr(), D[off].data_ptr(),
                          F[off].data_ptr(), st.cuda_stream, sets_ptr=sets_ptr)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return spread(ts)

    res = {"tool": "stations_bench", **gpu_info(), "forward_config": "F1", "rows": B, "eval": []}
    one = station_obs(1, 99)[0]
    c.config_obs(one)
    single = timed(lambda: call(0, B))
    for S, K in ((256, 64), (64, 256), (1024, 16)):
        dobs = station_obs(S, 100 + S)
        sets = torch.from_numpy(np.repeat(np.arange(S, dtype=np.int32), K)).to(dev)
        c.config_obs(dobs)
        grouped = timed(lambda: call(0, B, sets.data_ptr()))

        def per_station():
            for s in range(S):
                c.config_obs(dobs[s])
                call(s * K, K)
        seq = timed(per_station)
        res["eval"].append({"S": S, "K": K, "grouped": grouped, "per_station": seq, "one_set": single,
                            "speedup_per_station_over_grouped": seq["median_ms"] / grouped["median_ms"],
                            "set_lookup_cost": grouped["median_ms"] / single["median_ms"] - 1.0})

    # HMC: 16 stations x 64 chains, base sampler, fixed number of trajectories per chain
    Sh, Kh = 16, 64
    dobs = station_obs(Sh, 7)
    bounds = driver_bounds(x0)
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    ids = np.tile(np.arange(Kh), Sh)
    sets = np.repeat(np.arange(Sh), Kh)

    def hmc_grouped():
        c.config_obs(dobs)
        return c.hmc_run(0, ids, bounds, sets=sets, **kw)["evals"]

    def hmc_seq():
        ev = 0
        for s in range(Sh):
            c.config_obs(dobs[s])
            ev += c.hmc_run(0, np.arange(Kh), bounds, **kw)["evals"]
        return ev
    hmc = {"S": Sh, "K": Kh, "max_iters": a.hmc_iters}
    for name, fn in (("grouped", hmc_grouped), ("per_station", hmc_seq)):
        fn()
        ts, evs = [], 0
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            evs = fn()
            ts.append(time.perf_counter() - t0)
        hmc[name] = {**spread(ts), "evals": int(evs), "evals_per_s": float(evs / np.median(ts))}
    hmc["speedup_per_station_over_grouped"] = hmc["per_station"]["median_ms"] / hmc["grouped"]["median_ms"]
    res["hmc"] = hmc
    c.close()
    line = json.dumps(res)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
