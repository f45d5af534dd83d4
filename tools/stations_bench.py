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
Leg "rays" (per-station ray parameters, rfs_config_obs_rays), every station with its own ray parameter:
  (d) F1 (S, K) = (256, 64), (1024, 16): the grouped call with a ray table vs the same grouped call with
      the shared ray parameter (two contexts, timed alternately, --inner calls per timing);
  (e) RF only, C3-like: n = 40, nt = 2048, three ray parameters per station, 65 536 models over 256
      stations, with a [256, 3] table vs the shared list (the propagate kernel dominates there).  The two
      contexts live side by side, so each gets a 48 GB workspace budget (RFS_WS_BUDGET_MB): both run the
      batch in the same two chunks;
  (f) HMC, 16 stations x 64 chains, distinct ray parameters: one grouped run vs 16 single-station runs,
      each in a context configured with its station's ray parameter.
Leg "periods" (per-station SWD period lists, rfs_config_obs_periods), every station observing a seeded
random contiguous window of 60-100 % of each of the lists tRc and tRg (chosen independently):
  (g) F1 joint, (S, K) = (256, 64), (1024, 16): the grouped call with the mask vs the same grouped call
      on the full grid (two contexts, timed alternately, --inner calls per timing) vs one context
      reconfigured for each station in turn (config_swd on its subset lists, config_obs, its K rows);
  (h) SWD only, n = 40, modes 0-2, 24 Rc and 18 Rg periods, 64 stations x 64 models: the same three;
  (i) HMC, 16 stations x 64 chains: one grouped run with the mask vs 16 single-station runs, each in a
      context configured on its station's subset lists.
Leg "rfwin" (per-station receiver-function samples, rfs_config_obs_rf_samples), every station fitting a
seeded window of 40-100 % of each trace, about a quarter of the stations missing one ray bin (three ray
parameters 0.045, 0.06, 0.075 in place of F1's one, so that a bin can be missing):
  (j) F1 joint, (S, K) = (256, 64), (1024, 16): the grouped call with the mask vs the same grouped call
      without a table (two contexts, timed alternately, --inner calls per timing);
  (k) RF only, frequency method, n = 40, nt = 2048, three rays, 256 stations x 256 models: the same two
      (48 GB workspace budget each, as in (e));
  (l) RF only, time method, F1 layers and sampling, 64 stations x 16 models: the same two;
  (m) HMC, 16 stations x 64 chains with whole-trace masks (missing bins only): one grouped run vs 16
      single-station runs, each in a context configured on its station's observed rays.
Leg "gauss" (per-station Gaussian widths, rfs_config_obs_gauss), every station with its own widths:
  (n) F1 joint, one width per station drawn from {1.0, 1.5, 2.0, 2.5, 3.0}, (S, K) = (256, 64), (1024, 16):
      the grouped call with the width table vs the same grouped call on the shared width (two contexts,
      timed alternately, --inner calls per timing) vs one context reconfigured for each station in turn
      (config_rf on its width, config_obs, its K rows);
  (o) RF only, frequency method, n = 40, nt = 2048, three rays, two widths per station, 256 stations x 256
      models: the table vs the shared widths (48 GB workspace budget each, as in (e));
  (p) RF only, time method, F1 layers and sampling, two widths per station, 64 stations x 16 models: the
      same two;
  (q) HMC, 16 stations x 64 chains: one grouped run vs 16 single-station runs, each in a context configured
      with its station's width.
--legs sets,rays,periods,rfwin,gauss selects the legs (default sets,rays); the legs run replace their keys in
--out and keep the others.
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
    ap.add_argument("--legs", default="sets,rays")
    ap.add_argument("--inner", type=int, default=20, help="calls per timing in the rays leg")
    a = ap.parse_args()
    legs = set(a.legs.split(","))
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

    res = {}
    if os.path.exists(a.out):
        with open(a.out) as f:
            res = json.loads(f.read())
    if "rays" in legs:
        res["rays"] = rays_leg(a, torch, station_obs, X, nd)
    if "periods" in legs:
        res["periods"] = periods_leg(a, torch, X)
    if "rfwin" in legs:
        res["rfwin"] = rfwin_leg(a, torch, X)
    if "gauss" in legs:
        res["gauss"] = gauss_leg(a, torch, X)
    if "sets" not in legs:
        c.close()
        return write(a, res)
    res.update({"tool": "stations_bench", **gpu_info(), "forward_config": "F1", "rows": B, "eval": []})
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
    write(a, res)


def write(a, res):
    line = json.dumps(res)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


def rays_leg(a, torch, station_obs, X, nd):
    """Per-station ray parameters against the shared one, same grouped call (see the module docstring)."""
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models
    from bench import layered_models
    cfg, x0 = f1_config(), f1_true_model()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    out = {**gpu_info(), "inner_calls": a.inner, "eval": []}

    def contexts(which, n, rays, nt, dt, gauss, dobs, table):
        """(shared, table): two contexts on the same stations, without and with the ray table"""
        cs = []
        for with_table in (False, True):
            c = Context(0)
            if which != 1:
                c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
            c.config_rf(n, rays, nt, dt, gauss, cfg["time_shift"], cfg["water"], "P", "freq")
            c.config_obs(dobs)
            if with_table:
                c.config_obs_rays(table)
            cs.append(c)
        return cs

    def alternate(cs, which, Xd, sets):
        B = Xd.shape[0]
        U = torch.empty(B, dtype=torch.float64, device=dev)
        G = torch.empty(Xd.shape, dtype=torch.float64, device=dev)
        D = torch.empty(B, cs[0].ndata(which), dtype=torch.float64, device=dev)
        F = torch.empty(B, dtype=torch.uint8, device=dev)

        def call(c):
            for _ in range(a.inner):
                c.misfit_grad_dev(B, Xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                                  st.cuda_stream, sets_ptr=sets.data_ptr())
        ts = ([], [])
        for c in cs:
            call(c)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for k, c in enumerate(cs):
                t0 = time.perf_counter()
                call(c)
                torch.cuda.synchronize()
                ts[k].append((time.perf_counter() - t0) / a.inner)
        for c in cs:
            c.close()
        shared, table = spread(ts[0]), spread(ts[1])
        return {"shared_ray": shared, "ray_table": table, "table_cost": table["median_ms"] / shared["median_ms"] - 1.0}

    rng = np.random.default_rng(17)
    for S, K in ((256, 64), (1024, 16)):
        dobs = station_obs(S, 100 + S)
        table = rng.uniform(0.04, 0.08, S)
        sets = torch.from_numpy(np.repeat(np.arange(S, dtype=np.int32), K)).to(dev)
        cs = contexts(0, x0.size // 2, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], dobs, table)
        out["eval"].append({"workload": "F1 joint, %d stations x %d models" % (S, K), "S": S, "K": K,
                            **alternate(cs, 0, X, sets)})
    # RF only, C3-like
    n, nt, S, K = 40, 2048, 256, 256
    rays = [0.04, 0.06, 0.08]
    Xc = torch.from_numpy(layered_models(S * K, n, 2)).to(dev)
    table = np.sort(rng.uniform(0.035, 0.085, (S, 3)), axis=1)
    dobs = 0.01 * np.random.default_rng(3).standard_normal((S, 3 * nt))
    sets = torch.from_numpy(np.repeat(np.arange(S, dtype=np.int32), K)).to(dev)
    old = os.environ.get("RFS_WS_BUDGET_MB")
    os.environ["RFS_WS_BUDGET_MB"] = "48000"
    try:
        cs = contexts(1, n, rays, nt, 0.05, 2.5, dobs, table)
    finally:
        if old is None:
            del os.environ["RFS_WS_BUDGET_MB"]
        else:
            os.environ["RFS_WS_BUDGET_MB"] = old
    out["rf_c3"] = {"workload": "RF only (freq), n=40, nt=2048, dt=0.05, a=2.5, three ray parameters per station, "
                                "%d stations x %d models" % (S, K), "S": S, "K": K, **alternate(cs, 1, Xc, sets)}
    # HMC, 16 stations x 64 chains, distinct ray parameters
    Sh, Kh = 16, 64
    dobs = station_obs(Sh, 7)
    table = np.linspace(0.04, 0.08, Sh)
    bounds = driver_bounds(x0)
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    n = x0.size // 2
    grouped = contexts(0, n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], dobs, table)
    grouped[0].close()
    single = []
    for s in range(Sh):
        c = Context(0)
        c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
        c.config_rf(n, float(table[s]), cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"], "P", "freq")
        c.config_obs(dobs[s])
        single.append(c)
    ids, hsets = np.tile(np.arange(Kh), Sh), np.repeat(np.arange(Sh), Kh)
    runs = {"grouped": lambda: grouped[1].hmc_run(0, ids, bounds, sets=hsets, **kw)["evals"],
            "per_station": lambda: sum(single[s].hmc_run(0, np.arange(Kh), bounds, **kw)["evals"] for s in range(Sh))}
    hmc = {"S": Sh, "K": Kh, "max_iters": a.hmc_iters}
    for name, fn in runs.items():
        fn()
        ts, evs = [], 0
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            evs = fn()
            ts.append(time.perf_counter() - t0)
        hmc[name] = {**spread(ts), "evals": int(evs), "evals_per_s": float(evs / np.median(ts))}
    hmc["speedup_per_station_over_grouped"] = hmc["per_station"]["median_ms"] / hmc["grouped"]["median_ms"]
    out["hmc"] = hmc
    grouped[1].close()
    for c in single:
        c.close()
    return out


def periods_leg(a, torch, X):
    """Per-station period lists against the full grid and against one context per station (see the
    module docstring)."""
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models
    cfg, x0 = f1_config(), f1_true_model()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    out = {**gpu_info(), "inner_calls": a.inner, "mask": "contiguous window of 60-100 % of each list", "eval": []}
    rng = np.random.default_rng(23)

    def masks(S, lists):
        rows = []
        for _ in range(S):
            parts = []
            for t in lists:
                k = int(rng.integers(int(np.ceil(0.6 * len(t))), len(t) + 1))
                o = int(rng.integers(0, len(t) - k + 1))
                m = np.zeros(len(t), dtype=bool)
                m[o:o + k] = True
                parts.append(m)
            rows.append(np.concatenate(parts))
        return np.array(rows)

    def configure(c, which, n, lists, modes):
        if which != 1:
            c.config_swd(n, *lists, mode=modes)
        if which != 2:
            c.config_rf(n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"], cfg["water"],
                        cfg["rf_type"], cfg["method"])

    def subset(lists, u):
        r, o = [], 0
        for t in lists:
            r.append(np.asarray(t)[u[o:o + len(t)]])
            o += len(t)
        return r

    def observations(which, n, lists, modes, x_true, S, seed):
        c = Context(0)
        configure(c, which, n, lists, modes)
        c.config_obs(np.zeros((S, c.ndata(which))))
        _, _, d, _ = c.misfit_grad_host(perturbed_models(x_true, S, seed=seed, rel=0.05), which, sets=np.arange(S))
        c.close()
        d = np.where(np.isfinite(d), d, 0.0)
        return d + 0.01 * np.random.default_rng(seed).standard_normal(d.shape)

    def compare(which, n, lists, modes, Xd, S, K, dobs, use):
        nt = cfg["nt"] if which == 0 else 0
        nm = int(np.size(modes))
        B = Xd.shape[0]
        sets = torch.from_numpy(np.repeat(np.arange(S, dtype=np.int32), K)).to(dev)
        cs = []
        for with_mask in (True, False):
            c = Context(0)
            configure(c, which, n, lists, modes)
            c.config_obs(dobs)
            if with_mask:
                c.config_obs_periods(use)
            cs.append(c)
        U = torch.empty(B, dtype=torch.float64, device=dev)
        G = torch.empty(Xd.shape, dtype=torch.float64, device=dev)
        D = torch.empty(B, cs[0].ndata(which), dtype=torch.float64, device=dev)
        F = torch.empty(B, dtype=torch.uint8, device=dev)

        def call(c):
            for _ in range(a.inner):
                c.misfit_grad_dev(B, Xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                                  st.cuda_stream, sets_ptr=sets.data_ptr())
        ts = ([], [])
        for c in cs:
            call(c)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for k, c in enumerate(cs):
                t0 = time.perf_counter()
                call(c)
                torch.cuda.synchronize()
                ts[k].append((time.perf_counter() - t0) / a.inner)
        for c in cs:
            c.close()
        # what a user does without the table: one context, reconfigured for each station in turn
        one = Context(0)
        configure(one, which, n, lists, modes)
        compact = [np.concatenate([dobs[s, :nt], dobs[s, nt:][np.tile(use[s], nm)]]) for s in range(S)]
        subs = [subset(lists, use[s]) for s in range(S)]

        def per_station():
            for s in range(S):
                one.config_swd(n, *subs[s], mode=modes)
                one.config_obs(compact[s])
                one.misfit_grad_dev(K, Xd[s * K].data_ptr(), which, U[s * K].data_ptr(), G[s * K].data_ptr(),
                                    D[s * K].data_ptr(), F[s * K].data_ptr(), st.cuda_stream)
        per_station()
        torch.cuda.synchronize()
        tp = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            per_station()
            torch.cuda.synchronize()
            tp.append(time.perf_counter() - t0)
        one.close()
        masked, grid, seq = spread(ts[0]), spread(ts[1]), spread(tp)
        return {"masked": masked, "full_grid": grid, "per_station": seq,
                "observed_share": float(use.mean()),
                "masked_over_full_grid": masked["median_ms"] / grid["median_ms"],
                "speedup_per_station_over_masked": seq["median_ms"] / masked["median_ms"]}

    n = x0.size // 2
    f1 = (cfg["tRc"], cfg["tRg"], [], [])
    for S, K in ((256, 64), (1024, 16)):
        dobs = observations(0, n, f1, 0, x0, S, 100 + S)
        use = masks(S, f1[:2])
        out["eval"].append({"workload": "F1 joint, %d stations x %d models" % (S, K), "S": S, "K": K,
                            **compare(0, n, f1, 0, X[:S * K], S, K, dobs, use)})
    # SWD only, n = 40, modes 0-2
    n40, S, K = 40, 64, 64
    lists = (np.geomspace(2, 100, 24), np.geomspace(3, 80, 18), [], [])
    i = np.arange(n40)
    x40 = np.hstack((2.0 + 2.7 * (i / (n40 - 1.0)) ** 0.7, np.hstack((0.5 + 0.1 * i[:-1], [0.0]))))
    X40 = torch.from_numpy(perturbed_models(x40, S * K, seed=31, rel=0.05)).to(dev)
    dobs = observations(2, n40, lists, [0, 1, 2], x40, S, 41)
    out["n40"] = {"workload": "SWD only, n=40, modes 0-2, 24 Rc + 18 Rg periods, %d stations x %d models" % (S, K),
                  "S": S, "K": K, **compare(2, n40, lists, [0, 1, 2], X40, S, K, dobs, masks(S, lists[:2]))}
    # HMC, 16 stations x 64 chains
    Sh, Kh = 16, 64
    dobs = observations(0, n, f1, 0, x0, Sh, 7)
    use = masks(Sh, f1[:2])
    bounds = driver_bounds(x0)
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    grouped = Context(0)
    configure(grouped, 0, n, f1, 0)
    grouped.config_obs(dobs)
    grouped.config_obs_periods(use)
    single = []
    for s in range(Sh):
        c = Context(0)
        configure(c, 0, n, subset(f1, use[s]), 0)
        c.config_obs(np.concatenate([dobs[s, :cfg["nt"]], dobs[s, cfg["nt"]:][use[s]]]))
        single.append(c)
    ids, hsets = np.tile(np.arange(Kh), Sh), np.repeat(np.arange(Sh), Kh)
    runs = {"grouped": lambda: grouped.hmc_run(0, ids, bounds, sets=hsets, **kw)["evals"],
            "per_station": lambda: sum(single[s].hmc_run(0, np.arange(Kh), bounds, **kw)["evals"] for s in range(Sh))}
    hmc = {"S": Sh, "K": Kh, "max_iters": a.hmc_iters}
    for name, fn in runs.items():
        fn()
        ts, evs = [], 0
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            evs = fn()
            ts.append(time.perf_counter() - t0)
        hmc[name] = {**spread(ts), "evals": int(evs), "evals_per_s": float(evs / np.median(ts))}
    hmc["speedup_per_station_over_grouped"] = hmc["per_station"]["median_ms"] / hmc["grouped"]["median_ms"]
    out["hmc"] = hmc
    grouped.close()
    for c in single:
        c.close()
    return out


def rfwin_leg(a, torch, X):
    """Per-station RF samples against the same grouped call without a table, and the HMC against one
    context per station on its observed rays (see the module docstring)."""
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models
    from bench import layered_models
    cfg, x0 = f1_config(), f1_true_model()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    rays = [0.045, 0.06, 0.075]
    out = {**gpu_info(), "inner_calls": a.inner, "rays": rays,
           "mask": "window of 40-100 % of each trace, a quarter of the stations miss one ray bin", "eval": []}
    rng = np.random.default_rng(29)

    def masks(S, nt, whole=False):
        u = np.zeros((S, len(rays), nt), dtype=bool)
        for s in range(S):
            for r in range(len(rays)):
                k = nt if whole else int(rng.integers(int(np.ceil(0.4 * nt)), nt + 1))
                o = int(rng.integers(0, nt - k + 1))
                u[s, r, o:o + k] = True
            if rng.random() < 0.25:
                u[s, int(rng.integers(0, len(rays)))] = False
        return u.reshape(S, -1)

    def configure(c, which, n, nt, dt, gauss, method, rp=rays):
        if which != 1:
            c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
        c.config_rf(n, rp, nt, dt, gauss, cfg["time_shift"], cfg["water"], "P", method)

    def observations(which, n, nt, dt, gauss, method, Xs):
        c = Context(0)
        configure(c, which, n, nt, dt, gauss, method)
        S = Xs.shape[0]
        c.config_obs(np.zeros((S, c.ndata(which))))
        _, _, d, _ = c.misfit_grad_host(Xs, which, sets=np.arange(S))
        c.close()
        d = np.where(np.isfinite(d), d, 0.0)
        return d + 0.01 * np.random.default_rng(S).standard_normal(d.shape)

    def compare(which, n, nt, dt, gauss, method, Xd, S, K, dobs, use):
        B = Xd.shape[0]
        sets = torch.from_numpy(np.repeat(np.arange(S, dtype=np.int32), K)).to(dev)
        cs = []
        for with_mask in (True, False):
            c = Context(0)
            configure(c, which, n, nt, dt, gauss, method)
            c.config_obs(dobs)
            if with_mask:
                c.config_obs_rf_samples(use)
            cs.append(c)
        U = torch.empty(B, dtype=torch.float64, device=dev)
        G = torch.empty(Xd.shape, dtype=torch.float64, device=dev)
        D = torch.empty(B, cs[0].ndata(which), dtype=torch.float64, device=dev)
        F = torch.empty(B, dtype=torch.uint8, device=dev)

        def call(c):
            for _ in range(a.inner):
                c.misfit_grad_dev(B, Xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                                  st.cuda_stream, sets_ptr=sets.data_ptr())
        ts = ([], [])
        for c in cs:
            call(c)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for k, c in enumerate(cs):
                t0 = time.perf_counter()
                call(c)
                torch.cuda.synchronize()
                ts[k].append((time.perf_counter() - t0) / a.inner)
        for c in cs:
            c.close()
        masked, plain = spread(ts[0]), spread(ts[1])
        return {"masked": masked, "no_table": plain, "observed_share": float(use.mean()),
                "mask_cost": masked["median_ms"] / plain["median_ms"] - 1.0}

    n = x0.size // 2
    f1 = (n, cfg["nt"], cfg["dt"], cfg["gauss"])
    for S, K in ((256, 64), (1024, 16)):
        dobs = observations(0, *f1, "freq", perturbed_models(x0, S, seed=100 + S, rel=0.05))
        out["eval"].append({"workload": "F1 joint, three rays, %d stations x %d models" % (S, K), "S": S, "K": K,
                            **compare(0, *f1, "freq", X[:S * K], S, K, dobs, masks(S, cfg["nt"]))})
        progress(out["eval"][-1])
    # RF only, frequency method, C3-like
    nc, ntc, S, K = 40, 2048, 256, 256
    Xc = torch.from_numpy(layered_models(S * K, nc, 2)).to(dev)
    dobs = 0.01 * np.random.default_rng(3).standard_normal((S, 3 * ntc))
    old = os.environ.get("RFS_WS_BUDGET_MB")
    os.environ["RFS_WS_BUDGET_MB"] = "48000"
    try:
        out["rf_c3"] = {"workload": "RF only (freq), n=40, nt=2048, dt=0.05, a=2.5, three rays, "
                                    "%d stations x %d models" % (S, K), "S": S, "K": K,
                        **compare(1, nc, ntc, 0.05, 2.5, "freq", Xc, S, K, dobs, masks(S, ntc))}
    finally:
        if old is None:
            del os.environ["RFS_WS_BUDGET_MB"]
        else:
            os.environ["RFS_WS_BUDGET_MB"] = old
    progress(out["rf_c3"])
    # RF only, time method
    S, K = 64, 16
    dobs = observations(1, *f1, "time", perturbed_models(x0, S, seed=43, rel=0.05))
    out["rf_time"] = {"workload": "RF only (time), F1 layers and sampling, three rays, %d stations x %d models"
                                  % (S, K), "S": S, "K": K,
                      **compare(1, *f1, "time", X[:S * K], S, K, dobs, masks(S, cfg["nt"]))}
    progress(out["rf_time"])
    # HMC, 16 stations x 64 chains, whole-trace masks
    Sh, Kh = 16, 64
    dobs = observations(0, *f1, "freq", perturbed_models(x0, Sh, seed=7, rel=0.05))
    use = masks(Sh, cfg["nt"], whole=True)
    bounds = driver_bounds(x0)
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    grouped = Context(0)
    configure(grouped, 0, *f1, "freq")
    grouped.config_obs(dobs)
    grouped.config_obs_rf_samples(use)
    single = []
    for s in range(Sh):
        obs = use[s].reshape(len(rays), -1).all(axis=1)
        c = Context(0)
        configure(c, 0, *f1, "freq", np.asarray(rays)[obs].tolist())
        c.config_obs(np.concatenate([dobs[s, :use.shape[1]][use[s]], dobs[s, use.shape[1]:]]))
        single.append(c)
    ids, hsets = np.tile(np.arange(Kh), Sh), np.repeat(np.arange(Sh), Kh)
    runs = {"grouped": lambda: grouped.hmc_run(0, ids, bounds, sets=hsets, **kw)["evals"],
            "per_station": lambda: sum(single[s].hmc_run(0, np.arange(Kh), bounds, **kw)["evals"] for s in range(Sh))}
    hmc = {"S": Sh, "K": Kh, "max_iters": a.hmc_iters, "stations_missing_a_bin": int((~use.all(axis=1)).sum())}
    for name, fn in runs.items():
        fn()
        ts, evs = [], 0
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            evs = fn()
            ts.append(time.perf_counter() - t0)
        hmc[name] = {**spread(ts), "evals": int(evs), "evals_per_s": float(evs / np.median(ts))}
    hmc["speedup_per_station_over_grouped"] = hmc["per_station"]["median_ms"] / hmc["grouped"]["median_ms"]
    out["hmc"] = hmc
    grouped.close()
    for c in single:
        c.close()
    return out


def gauss_leg(a, torch, X):
    """Per-station Gaussian widths against the same grouped call on the shared widths, and against one
    context reconfigured per station (see the module docstring)."""
    from rfsurfhmc_b200._lib import Context
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, perturbed_models
    from bench import layered_models
    cfg, x0 = f1_config(), f1_true_model()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev)
    widths = np.array([1.0, 1.5, 2.0, 2.5, 3.0])
    out = {**gpu_info(), "inner_calls": a.inner, "widths": widths.tolist(), "eval": []}
    rng = np.random.default_rng(31)

    def configure(c, which, n, rays, nt, dt, gauss, method):
        if which != 1:
            c.config_swd(n, tRc=cfg["tRc"], tRg=cfg["tRg"])
        c.config_rf(n, rays, nt, dt, gauss, cfg["time_shift"], cfg["water"], "P", method)

    def observations(which, shape, table, Xs):
        c = Context(0)
        configure(c, which, *shape)
        S = Xs.shape[0]
        c.config_obs(np.zeros((S, c.ndata(which))))
        c.config_obs_gauss(table)
        _, _, d, _ = c.misfit_grad_host(Xs, which, sets=np.arange(S))
        c.close()
        d = np.where(np.isfinite(d), d, 0.0)
        return d + 0.01 * np.random.default_rng(S).standard_normal(d.shape)

    def compare(which, shape, Xd, S, K, dobs, table, per_station=False):
        B = Xd.shape[0]
        sets = torch.from_numpy(np.repeat(np.arange(S, dtype=np.int32), K)).to(dev)
        cs = []
        for with_table in (True, False):
            c = Context(0)
            configure(c, which, *shape)
            c.config_obs(dobs)
            if with_table:
                c.config_obs_gauss(table)
            cs.append(c)
        U = torch.empty(B, dtype=torch.float64, device=dev)
        G = torch.empty(Xd.shape, dtype=torch.float64, device=dev)
        D = torch.empty(B, cs[0].ndata(which), dtype=torch.float64, device=dev)
        F = torch.empty(B, dtype=torch.uint8, device=dev)

        def call(c):
            for _ in range(a.inner):
                c.misfit_grad_dev(B, Xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), F.data_ptr(),
                                  st.cuda_stream, sets_ptr=sets.data_ptr())
        ts = ([], [])
        for c in cs:
            call(c)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for k, c in enumerate(cs):
                t0 = time.perf_counter()
                call(c)
                torch.cuda.synchronize()
                ts[k].append((time.perf_counter() - t0) / a.inner)
        for c in cs:
            c.close()
        tab, shared = spread(ts[0]), spread(ts[1])
        r = {"width_table": tab, "shared_width": shared, "table_cost": tab["median_ms"] / shared["median_ms"] - 1.0}
        if not per_station:
            return r
        # what a user does without the table: one context, reconfigured for each station in turn
        one = Context(0)
        n, rays, nt, dt = shape[:4]

        def seq():
            for s in range(S):
                one.config_rf(n, rays, nt, dt, float(table[s]), cfg["time_shift"], cfg["water"], "P", shape[-1])
                one.config_obs(dobs[s])
                one.misfit_grad_dev(K, Xd[s * K].data_ptr(), which, U[s * K].data_ptr(), G[s * K].data_ptr(),
                                    D[s * K].data_ptr(), F[s * K].data_ptr(), st.cuda_stream)
        configure(one, which, *shape)
        seq()
        torch.cuda.synchronize()
        tp = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            seq()
            torch.cuda.synchronize()
            tp.append(time.perf_counter() - t0)
        one.close()
        r["per_station"] = spread(tp)
        r["speedup_per_station_over_table"] = r["per_station"]["median_ms"] / tab["median_ms"]
        return r

    n = x0.size // 2
    f1 = (n, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], "freq")
    for S, K in ((256, 64), (1024, 16)):
        table = rng.choice(widths, S)
        dobs = observations(0, f1, table, perturbed_models(x0, S, seed=100 + S, rel=0.05))
        out["eval"].append({"workload": "F1 joint, one width per station, %d stations x %d models" % (S, K),
                            "S": S, "K": K, **compare(0, f1, X[:S * K], S, K, dobs, table, per_station=True)})
        progress(out["eval"][-1])
    # RF only, frequency method, C3-like, two widths per station
    nc, ntc, S, K = 40, 2048, 256, 256
    c3 = (nc, [0.04, 0.06, 0.08], ntc, 0.05, [1.0, 2.5], "freq")
    Xc = torch.from_numpy(layered_models(S * K, nc, 2)).to(dev)
    table = np.sort(rng.choice(widths, (S, 2)), axis=1)
    dobs = 0.01 * np.random.default_rng(3).standard_normal((S, 3 * 2 * ntc))
    old = os.environ.get("RFS_WS_BUDGET_MB")
    os.environ["RFS_WS_BUDGET_MB"] = "48000"
    try:
        out["rf_c3"] = {"workload": "RF only (freq), n=40, nt=2048, dt=0.05, three rays, two widths per station, "
                                    "%d stations x %d models" % (S, K), "S": S, "K": K,
                        **compare(1, c3, Xc, S, K, dobs, table)}
    finally:
        if old is None:
            del os.environ["RFS_WS_BUDGET_MB"]
        else:
            os.environ["RFS_WS_BUDGET_MB"] = old
    progress(out["rf_c3"])
    # RF only, time method, two widths per station
    S, K = 64, 16
    ft = (n, cfg["ray_p"], cfg["nt"], cfg["dt"], [1.0, 2.5], "time")
    table = np.sort(rng.choice(widths, (S, 2)), axis=1)
    dobs = observations(1, ft, table, perturbed_models(x0, S, seed=43, rel=0.05))
    out["rf_time"] = {"workload": "RF only (time), F1 layers and sampling, two widths per station, "
                                  "%d stations x %d models" % (S, K), "S": S, "K": K,
                      **compare(1, ft, X[:S * K], S, K, dobs, table)}
    progress(out["rf_time"])
    # HMC, 16 stations x 64 chains, base sampler
    Sh, Kh = 16, 64
    table = rng.choice(widths, Sh)
    dobs = observations(0, f1, table, perturbed_models(x0, Sh, seed=7, rel=0.05))
    bounds = driver_bounds(x0)
    kw = dict(dt=0.1, Lrange=(5, 20), seed=991206, nsamples=a.hmc_iters + 1, ndraws=0, max_iters=a.hmc_iters,
              want_samples=False)
    grouped = Context(0)
    configure(grouped, 0, *f1)
    grouped.config_obs(dobs)
    grouped.config_obs_gauss(table)
    single = []
    for s in range(Sh):
        c = Context(0)
        configure(c, 0, n, cfg["ray_p"], cfg["nt"], cfg["dt"], float(table[s]), "freq")
        c.config_obs(dobs[s])
        single.append(c)
    ids, hsets = np.tile(np.arange(Kh), Sh), np.repeat(np.arange(Sh), Kh)
    runs = {"grouped": lambda: grouped.hmc_run(0, ids, bounds, sets=hsets, **kw)["evals"],
            "per_station": lambda: sum(single[s].hmc_run(0, np.arange(Kh), bounds, **kw)["evals"] for s in range(Sh))}
    hmc = {"S": Sh, "K": Kh, "max_iters": a.hmc_iters}
    for name, fn in runs.items():
        fn()
        ts, evs = [], 0
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            evs = fn()
            ts.append(time.perf_counter() - t0)
        hmc[name] = {**spread(ts), "evals": int(evs), "evals_per_s": float(evs / np.median(ts))}
    hmc["speedup_per_station_over_grouped"] = hmc["per_station"]["median_ms"] / hmc["grouped"]["median_ms"]
    out["hmc"] = hmc
    grouped.close()
    for c in single:
        c.close()
    return out


def progress(r):
    """One finished workload of a leg on stderr (the RF C3 workloads take minutes)."""
    print(json.dumps(r), file=sys.stderr, flush=True)


if __name__ == "__main__":
    main()
