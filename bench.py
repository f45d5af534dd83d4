#!/usr/bin/env python
"""bench.py — joint RF+SWD forward+gradient evaluations/s on N B200s (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W            (our arm: sm_100a CUDA through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  (CPU arm: oracle restatement of the
                                                              reference, all host threads)
    torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, chains sharded)

One "step" = one batched Joint_RF_SWD.misfit_and_grad over `--chains` chain states per GPU at the
C1/C4 sizes of SURVEY.md §8 (n=7 layers, 36 Rc + 36 Rg periods, RF nt=125 -> nft=128; reference
param.yaml), i.e. the evaluation every leapfrog step of every chain performs.  Prints ONE JSON line.

Everything on the value path is measured in this run: the per-kernel times behind `roofline` /
`kernels` come from CUDA events around every launch (rfs_profile_eval), the secular-evaluation count
from a device counter, the FP64 peak from a DFMA micro-benchmark.  Only `traffic` (DRAM bytes of an
`ncu --set full` capture) is read from profiles/ — ncu cannot run inside a timed bench.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# frozen algorithmic-work constants (BASELINE.md §3, hand counts of SURVEY.md §8d); 1 FMA = 2 flop
F_R = 375.0      # flop per Rayleigh secular-function layer step (dltar4 body)
E_R = 3500.0     # flop per layer per (T, c): Rayleigh eigenfunctions + energy integrals + kernels
P_RF = 2900.0    # flop per (frequency bin, layer): RF propagator + 4 derivative matrices + O(n) products
N_LAYERS = 7


def workload(nchains, seed):
    from rfsurfhmc_b200.fixtures import f1_config, f1_true_model, driver_bounds, sorted_uniform_models
    cfg = f1_config()
    x0 = f1_true_model()
    X = sorted_uniform_models(driver_bounds(x0), nchains, seed)
    return cfg, x0, X


def layered_models(B, n, seed, thk0=None, jitter=0.04):
    """synthetic n-layer crust of SURVEY.md §8d (configs 2, 3, 5)"""
    rng = np.random.default_rng(seed)
    if thk0 is None:
        thk0 = np.hstack((0.5 + 0.1 * np.arange(n - 1), [0.0]))
    thk = thk0[None, :] * (1 + 0.1 * rng.uniform(-1, 1, (B, n)))
    thk[:, -1] = 0.0
    vs0 = 2.0 + 2.7 * (np.arange(n) / (n - 1.0))**0.7
    vs = np.clip(vs0[None, :] * (1 + jitter * rng.standard_normal((B, n))), 1.5, 5.0)
    return np.hstack((vs, thk))


def make_dobs(cfg, x0):
    """CPU arm only: observations = synthetics of the true model (main_base.py:49-56) from the
    oracle, which is the implementation that arm measures."""
    from oracle.oracle import Oracle
    O = Oracle()
    nd = cfg["nt"] + len(cfg["tRc"]) + len(cfg["tRg"])
    _, _, d, _ = O.joint_batch(x0[None, :], np.zeros(nd), cfg)
    return d[0]


def make_dobs_gpu(ctx, cfg, x0):
    """Our arm: observations = synthetics of the true model computed by the CUDA path itself, as
    the reference driver does with its own forward model (main_base.py:49-56)."""
    nd = cfg["nt"] + len(cfg["tRc"]) + len(cfg["tRg"])
    ctx.config_obs(np.zeros(nd))
    _, _, d, f = ctx.misfit_grad_host(x0[None, :])
    assert f[0]
    return d[0].copy()


class ClockSampler(threading.Thread):
    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev = dev
        self.rows = []
        self.stop = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons}


def cpu_arm(cfg, dobs, X, seconds, nthreads, which=0):
    """Oracle restatement (-O3 build) timed on the host cores: evaluations/s."""
    from oracle.oracle import Oracle
    O = Oracle(fast=True)
    chunk = max(64, 16 * nthreads)
    chunk = min(chunk, len(X))
    done = 0
    t0 = time.perf_counter()
    i = 0
    while True:
        xb = X[(i * chunk) % len(X):][:chunk]
        if len(xb) < chunk:
            xb = X[:chunk]
        O.joint_batch(xb, dobs, cfg, which=which, nthreads=nthreads)
        done += len(xb)
        i += 1
        if time.perf_counter() - t0 >= seconds:
            break
    dt = time.perf_counter() - t0
    return done / dt, done, dt


# --------------------------------------------------------------------------------------------------
# secondary workloads of BASELINE.json (configs[1], [2], [4]): one objective per chain, device-resident
# --------------------------------------------------------------------------------------------------
def _timed_eval(torch, ctx, xd, which, nd, reps=1):
    dev = xd.device
    B, n2 = xd.shape
    U = torch.empty(B, dtype=torch.float64, device=dev)
    G = torch.empty(B, n2, dtype=torch.float64, device=dev)
    D = torch.empty(B, nd, dtype=torch.float64, device=dev)
    Fl = torch.empty(B, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()

    def call():
        ctx.misfit_grad_dev(B, xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), Fl.data_ptr(),
                            st.cuda_stream)
    call()                                   # warm-up (allocates the workspace)
    torch.cuda.synchronize()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        call()
    e1.record(st)
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / reps
    prof = ctx.profile_eval(B, xd.data_ptr(), which, U.data_ptr(), G.data_ptr(), D.data_ptr(), Fl.data_ptr(),
                            st.cuda_stream)
    return sec, int((Fl == 0).sum().item()), (ctx.launches - l0) // max(1, reps), prof, (U, G, D, Fl)


def _kernel_table(prof):
    tot = sum(v[0] for v in prof.values())
    return {k: {"ms": round(v[0], 4), "launches": v[1], "share": round(v[0] / tot, 4) if tot else None}
            for k, v in prof.items() if v[1] > 0}


def config_legs(torch, dev_index, ncores, hbm_peak, fp64_peak, with_cpu=True):
    """C2, C3 (freq + time), C5 throughput on one GPU, each with its own bounded CPU baseline."""
    from rfsurfhmc_b200._lib import Context
    from oracle.oracle import Oracle
    dev = torch.device("cuda", dev_index)
    out = {}
    O = Oracle(fast=True) if with_cpu else None

    # ---- C2: SWD-only forward+Frechet, n=40, 60 periods, Rc+Rg+Lc+Lg, modes 0-2 in ONE objective
    n, B = 40, 65536
    T = np.geomspace(2, 100, 60)
    X = layered_models(B, n, 2)
    ctx = Context(dev_index)
    ctx.config_swd(n, T, T, T, T, mode=[0, 1, 2])
    nd = 720
    ctx.config_obs(np.full(nd, 3.0))
    xd = torch.from_numpy(X).to(dev)
    sec, nfail, nl, prof, _ = _timed_eval(torch, ctx, xd, 2, nd)
    leg = {"workload": "C2 SWD-only forward+Frechet objective: n=40, 60 periods, Rc+Rg+Lc+Lg, modes 0,1,2 as one "
                       "objective (720 data), batch %d" % B,
           "value": B / sec, "unit": "models/s", "seconds": sec, "failed_models": nfail, "gpu_launches": nl,
           "kernels": _kernel_table(prof), "root_search_mapping": list(ctx.last_roots_team())}
    if with_cpu:
        Xc = X[:96 * ncores]
        base = dict(tRc=T, tRg=T, tLc=T, tLg=T, ray_p=0.06, nt=64, dt=0.1, gauss=2.5, time_shift=5.0)
        t0 = time.perf_counter()
        for mode in (0, 1, 2):
            O.joint_batch(Xc, np.full(240, 3.0), dict(base, mode=mode), which=2, nthreads=ncores)
        tc = time.perf_counter() - t0
        leg["cpu_baseline"] = {"value": len(Xc) / tc, "unit": "models/s", "cores": ncores, "kind": "port",
                               "sample": "%d models, modes 0,1,2 (three reference calls per model), %.1f s" % (len(Xc), tc)}
    out["C2"] = leg
    del ctx, xd

    # ---- C3: RF-only forward+Frechet, nt=2048, a=2.5, three ray parameters in ONE objective
    nt, rays = 2048, [0.04, 0.06, 0.08]
    ctx = Context(dev_index)
    ctx.config_rf(n, rays, nt, 0.05, 2.5, 5.0, 1e-3, "P", "freq")
    ctx.config_obs(np.zeros(3 * nt))
    xd = torch.from_numpy(X).to(dev)
    sec, nfail, nl, prof, _ = _timed_eval(torch, ctx, xd, 1, 3 * nt)
    n2 = nt // 2 + 1
    kt = _kernel_table(prof)
    # achieved HBM GB/s of the spectral stages (bytes that cross HBM per profiled call / kernel time)
    Bc = B  # profile call covers the whole batch (possibly in chunks)
    by_prop = Bc * 3 * (2 * n2 + 2 * n * n2) * 16.0
    by_dec = by_prop + Bc * 3 * (nt * 8.0 + 2 * n * 8.0)
    if "rf_propagate" in kt:
        kt["rf_propagate"]["hbm_gbs"] = by_prop / (kt["rf_propagate"]["ms"] * 1e-3) / 1e9
        kt["rf_propagate"]["fp64_frac"] = (Bc * 3.0 * n2 * n * P_RF / (kt["rf_propagate"]["ms"] * 1e-3) / 1e12
                                          / fp64_peak) if fp64_peak else None
    if "rf_decon" in kt:
        kt["rf_decon"]["hbm_gbs"] = by_dec / (kt["rf_decon"]["ms"] * 1e-3) / 1e9
        kt["rf_decon"]["hbm_frac"] = kt["rf_decon"]["hbm_gbs"] / hbm_peak
    leg = {"workload": "C3 RF-only forward+Frechet objective (freq, water level): n=40, nt=2048, dt=0.05, a=2.5, "
                       "ray parameters 0.04/0.06/0.08 as one objective (6144 data), batch %d" % B,
           "value": B / sec, "unit": "models/s", "seconds": sec, "gpu_launches": nl, "kernels": kt}
    if with_cpu:
        Xc = X[:20 * ncores]
        base = dict(nt=nt, dt=0.05, gauss=2.5, time_shift=5.0, water=1e-3, rf_type="P", method="freq")
        t0 = time.perf_counter()
        for p in rays[:1]:
            O.joint_batch(Xc, np.zeros(nt), dict(base, ray_p=p), which=1, nthreads=ncores)
        tc = (time.perf_counter() - t0) * 3.0
        leg["cpu_baseline"] = {"value": len(Xc) / tc, "unit": "models/s", "cores": ncores, "kind": "port",
                               "sample": "%d models, one of the three ray parameters timed (x3), reference O(n^2) "
                                         "Frechet algorithm, %.1f s" % (len(Xc), tc / 3.0)}
    out["C3_freq"] = leg
    # time-domain method (iterative deconvolution of the trace and of all 4n Frechet traces)
    Bt = 1024
    ctx.config_rf(n, 0.06, nt, 0.05, 2.5, 5.0, 1e-3, "P", "time")
    ctx.config_obs(np.zeros(nt))
    xt = xd[:Bt].contiguous()
    sec, nfail, nl, prof, _ = _timed_eval(torch, ctx, xt, 1, nt)
    out["C3_time"] = {"workload": "C3 RF-only forward+Frechet objective, time-domain (iterative) deconvolution: n=40, "
                                  "nt=2048, one ray parameter, batch %d (161 deconvolutions per model)" % Bt,
                      "value": Bt / sec, "unit": "models/s", "seconds": sec, "gpu_launches": nl,
                      "kernels": _kernel_table(prof)}
    # forward only, time domain, at the full batch (one deconvolution per model)
    vs, thk = X[:, :n], X[:, n:]
    from oracle.oracle import brocher
    vp, rho = brocher(vs)
    q = np.full_like(vs, 9999.)
    ctx.rf_forward(thk[:256], rho[:256], vp[:256], vs[:256], q[:256], q[:256], 0.06, nt, 0.05, 2.5, 5.0,
                   method="time", rf_type="P")
    t0 = time.perf_counter()
    ctx.rf_forward(thk, rho, vp, vs, q, q, 0.06, nt, 0.05, 2.5, 5.0, method="time", rf_type="P")
    tf = time.perf_counter() - t0
    out["C3_time"]["forward_only"] = {"value": B / tf, "unit": "models/s", "batch": B,
                                      "note": "librf.forward drop-in (host buffers in and out)"}
    if with_cpu:
        Xc = X[:ncores]
        t0 = time.perf_counter()
        O.joint_batch(Xc, np.zeros(nt), dict(nt=nt, dt=0.05, gauss=2.5, time_shift=5.0, water=1e-3, rf_type="P",
                                             method="time", ray_p=0.06), which=1, nthreads=ncores)
        tc = time.perf_counter() - t0
        out["C3_time"]["cpu_baseline"] = {"value": len(Xc) / tc, "unit": "models/s", "cores": ncores, "kind": "port",
                                          "sample": "%d models, %.1f s" % (len(Xc), tc)}
    del ctx, xd, xt

    # ---- C5: fine parameterisation joint evaluation, 8192 chains per GPU
    n, B = 200, 8192
    T = np.geomspace(1, 150, 128)
    nt = 4096
    X = layered_models(B, n, 5, thk0=np.hstack((np.full(n - 1, 0.4), [0.0])))
    ctx = Context(dev_index)
    ctx.config_swd(n, T, T)
    ctx.config_rf(n, 0.06, nt, 0.025, 2.5, 5.0, 1e-3, "P", "freq")
    nd = nt + 256
    ctx.config_obs(np.hstack((np.zeros(nt), np.full(256, 3.3))))
    xd = torch.from_numpy(X).to(dev)
    sec, nfail, nl, prof, res = _timed_eval(torch, ctx, xd, 0, nd)
    leg = {"workload": "C5 joint RF+SWD evaluation: n=200 layers, 128 Rc + 128 Rg periods, RF nt=4096, %d chain "
                       "states on one GPU" % B,
           "value": B / sec, "unit": "evals/s", "seconds": sec, "failed_models": nfail, "gpu_launches": nl,
           "finite_grad_fraction": float(torch.isfinite(res[1]).all(dim=1).float().mean().item()),
           "kernels": _kernel_table(prof), "root_search_mapping": list(ctx.last_roots_team())}
    if with_cpu:
        Xc = X[:40 * ncores]
        cfg5 = dict(tRc=T, tRg=T, ray_p=0.06, nt=256, dt=0.025 * 16, gauss=2.5, time_shift=5.0, water=1e-3,
                    rf_type="P", method="freq")
        t0 = time.perf_counter()
        O.joint_batch(Xc, np.full(256, 3.3), cfg5, which=2, nthreads=ncores)
        t_swd = time.perf_counter() - t0
        Xr = X[:ncores]
        t0 = time.perf_counter()
        O.joint_batch(Xr, np.zeros(256), cfg5, which=1, nthreads=ncores)
        t_rf = (time.perf_counter() - t0) * (2049.0 / 129.0)
        per_model = t_swd / len(Xc) + t_rf / len(Xr)
        leg["cpu_baseline"] = {"value": 1.0 / per_model, "unit": "evals/s", "cores": ncores, "kind": "port",
                               "sample": "SWD part: %d models at full size (%.1f s); RF part: %d models on 129 of the "
                                         "2049 frequency bins (nt=256), time scaled by 2049/129 (the reference's "
                                         "O(n^2) Frechet pass needs minutes per model at n=200)"
                                         % (len(Xc), t_swd, len(Xr))}
    out["C5"] = leg
    return out


def dump_outputs(outdir, tensors, limit=64 * 10**6):
    """Per-chain outputs of one step as DIR/<name>.npy (flag as float32, the rest float64), so that two
    builds can be compared output for output on the same seeded inputs.  Above `limit` bytes in all, the
    same fixed, seeded sample of chains is kept from every array and its indices go to rows.npy.  Rows
    whose flag is 0 (failed root search) hold unspecified values."""
    arrays = {k: t.cpu().numpy().astype(np.float32 if t.dtype.itemsize == 1 else np.float64)
              for k, t in tensors.items()}
    nrows = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes for a in arrays.values()) / nrows
    if nrows * row_bytes > limit:
        keep = int((limit - 4096) // (row_bytes + 8))     # 4096: room for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(nrows, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(outdir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(outdir, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=16384, help="chain states per GPU (C4: 16384)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hmc", action="store_true", help="skip the device-resident HMC legs")
    ap.add_argument("--no-configs", action="store_true", help="skip the C2/C3/C5 legs (run at N=1 only)")
    ap.add_argument("--hmc-traj", type=int, default=100, help="trajectories per chain in the HMC legs")
    ap.add_argument("--da-budget", type=float, default=15.0, help="wall-clock budget of the uncapped DA leg (s)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write U, grad, dsyn and flag of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = os.cpu_count() or 1
    config = {"workload": "C4/C1 joint RF+SWD misfit_and_grad: n=7 layers, 36 Rc + 36 Rg periods (5-40 s), "
                          "RF nt=125 (nft=128) freq-domain P, %d chain states per GPU" % args.chains,
              "chains_per_gpu": args.chains, "parallelism": "chains sharded, no data-path collective",
              "l2": "inputs rotated over 4 batches + 256 MiB L2 flush between steps (inside the timed region), "
                    "in the device-resident loop and in the e2e loop alike"}

    # ------------------------------------------------------------------ reference (CPU) arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        cfg, x0, X = workload(4096, 1234)
        dobs = make_dobs(cfg, x0)
        per_step = max(1.0, min(10.0, 120.0 / max(1, args.steps + args.warmup)))
        for _ in range(min(args.warmup, 1)):
            cpu_arm(cfg, dobs, X, 0.5, ncores)
        tot, tt = 0, 0.0
        for _ in range(args.steps):
            v, done, dt = cpu_arm(cfg, dobs, X, per_step, ncores)
            tot += done
            tt += dt
        val = tot / tt
        print(json.dumps({
            "impl": "reference", "metric": "joint RF+SWD forward+gradient evaluations/s",
            "value": val, "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": val, "unit": "evals/s", "cores": ncores, "kind": "port",
                             "sample": "%d evaluations in %.1f s (oracle restatement of the reference CPU "
                                       "path, g++ -O3, %d threads; reference itself not buildable: no "
                                       "gfortran/FFTW3)" % (tot, tt, ncores)},
            "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return 0

    # ------------------------------------------------------------------ our arm
    # the contract is ONE line on stdout: library chatter (e.g. "NCCL version ...") goes to stderr
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from rfsurfhmc_b200._lib import Context
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (rfsurfhmc_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.chains
    cfg, x0, _ = workload(1, 0)
    ctx = Context(local_rank)
    ctx.config_swd(N_LAYERS, tRc=cfg["tRc"], tRg=cfg["tRg"])
    ctx.config_rf(N_LAYERS, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"],
                  cfg["water"], cfg["rf_type"], cfg["method"])
    dobs = make_dobs_gpu(ctx, cfg, x0)
    nd = dobs.size
    ctx.config_obs(dobs)
    nrot = 4
    Xs = [workload(B, 1000 + 97 * rank + i)[2] for i in range(nrot)]
    xd = [torch.from_numpy(x).to(dev) for x in Xs]
    U = torch.empty(B, dtype=torch.float64, device=dev)
    G = torch.empty(B, 2 * N_LAYERS, dtype=torch.float64, device=dev)
    D = torch.empty(B, nd, dtype=torch.float64, device=dev)
    Fl = torch.empty(B, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    def step(i, c=ctx, x=None, nb=B):
        flush.zero_()
        c.misfit_grad_dev(nb, (x if x is not None else xd[i % nrot]).data_ptr(), 0, U.data_ptr(), G.data_ptr(),
                          D.data_ptr(), Fl.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(nsteps, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(nsteps):
            step(i, **kw)
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1)

    for i in range(args.warmup):
        step(i)
    barrier()
    fp64_peak = ctx.measure_fp64_peak()
    ctx.count_evals(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launches
    ms = timed_steps(args.steps)
    if args.dump_outputs and rank == 0:       # before profile_eval below overwrites the buffers
        dump_outputs(args.dump_outputs, {"U": U, "grad": G, "dsyn": D, "flag": Fl})
    launches = ctx.launches - l0
    nev = ctx.read_evals()
    ctx.count_evals(False)
    n_fail = int((Fl == 0).sum().item())
    mapping_main = ctx.last_roots_team()
    sorted_main = ctx.last_roots_sched()

    # ---- per-kernel timing, live: CUDA events around every launch of one evaluation (RF branch
    # serialised for these calls so that each kernel is timed alone), median of 5 calls
    profs = []
    for i in range(5):
        flush.zero_()
        profs.append(ctx.profile_eval(B, xd[i % nrot].data_ptr(), 0, U.data_ptr(), G.data_ptr(), D.data_ptr(),
                                      Fl.data_ptr(), stream.cuda_stream))
    kms = {k: float(np.median([p[k][0] for p in profs])) for k in profs[0]}
    klaunch = {k: profs[0][k][1] for k in profs[0]}

    # ---- strong scaling (BASELINE config 4 wording: 16 384 chains sharded across 1/2/4/8 GPUs)
    strong = None
    if world > 1:
        Bs = max(1, 16384 // world)
        xs_ = xd[0][:Bs].contiguous()
        for i in range(3):
            step(i, x=xs_, nb=Bs)
        ms_s = timed_steps(args.steps, x=xs_, nb=Bs)
        strong = [ms_s, Bs, ctx.last_roots_team()]

    # ---- e2e: the public host-buffer API (rfsurfhmc_b200.batched.HostPipeline): every step copies
    # its inputs from pinned host memory and reads U, grad, dsyn, flag back to the host; the two
    # slots overlap the copies of one batch with the kernels of the next
    from rfsurfhmc_b200.batched import HostPipeline
    xh = [torch.from_numpy(x).pin_memory() for x in Xs]
    pipe = HostPipeline(cfg, dobs, N_LAYERS, B, device=local_rank)
    for i in range(3):
        pipe.submit(xh[i % nrot])
    pipe.drain()
    barrier()
    l_e2e0 = pipe.launches
    t0 = time.perf_counter()
    chk = 0.0
    for i in range(args.steps):
        flush.zero_()                       # same cache policy as the device-resident loop
        done = pipe.submit(xh[i % nrot])
        if done is not None:
            chk += float(done[0][0])        # the step's result is read on the host
    last = pipe.drain()
    chk += float(last[0][0])
    barrier()
    t_e2e = time.perf_counter() - t0
    launches_e2e = pipe.launches - l_e2e0
    sampler.stop = True
    del pipe

    # ---- device-resident HMC legs
    hmc = None
    if not args.no_hmc:
        from rfsurfhmc_b200.fixtures import driver_bounds
        from rfsurfhmc_b200 import distributed as Dm
        bounds = driver_bounds(x0)
        ntraj = args.hmc_traj

        def run_leg(total_chains, sampler_id, **kw):
            """chains sharded over the ranks; broadcast of the observations at start and NCCL all-gathers of
            the misfit history and the per-chain counters at the end are part of the leg (main_base.py:59-60,90)"""
            ids = Dm.shard_chains(total_chains, rank, world)
            barrier()
            t0 = time.perf_counter()
            d = Dm.bcast_array(dobs)
            ctx.config_obs(d)
            ho = ctx.hmc_run(sampler_id, ids, bounds, want_samples=False, want_syn=False, **kw)
            torch.cuda.synchronize()
            t1a = time.perf_counter()
            barrier()                      # ranks finish at different times: wait here, not inside the gather
            t1 = time.perf_counter()
            mis = Dm.gather_chains(ho["misfit"], total_chains)
            nit = Dm.gather_chains(ho["n_iter"], total_chains)
            nac = Dm.gather_chains(ho["n_acc"], total_chains)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            barrier()
            t3 = time.perf_counter()
            complete = int((ho["n_acc"] >= kw["nsamples"] + kw["ndraws"]).sum()) if kw.get("max_iters", 0) == 0 else None
            return {"t": t3 - t0, "t_gather": t2 - t1, "t_wait": t1 - t1a, "traj": float(nit.sum()), "acc": float(nac.sum()),
                    "evals": float(ho["evals"]), "steps": float(ho["global_steps"]), "chains": total_chains,
                    "misfit_shape": list(mis.shape), "complete_local": complete, "local_chains": len(ids)}

        legs = {}
        # C4 wording: 16 384 chains x L=20 leapfrog steps, sharded over the GPUs (strong scaling)
        legs["c4_strong"] = run_leg(16384, 0, dt=0.02, Lrange=(20, 20), seed=991206, nsamples=ntraj, ndraws=0,
                                    max_iters=ntraj)
        if world > 1:   # weak: the per-GPU batch of the headline
            legs["base_weak"] = run_leg(B * world, 0, dt=0.02, Lrange=(20, 20), seed=991206, nsamples=10, ndraws=0,
                                        max_iters=10)
        # C4 names the dual-averaging sampler (main_DA.py): lambda = L0*dt = 20*0.02, step size adapted
        # during the first half of the trajectories; L = int(lambda/dt) capped at 40 (extension, see
        # DESIGN.md: the reference's gamma = 0.05 lets L explode after one rejected warm-up trajectory)
        legs["da_capped"] = run_leg(B * world, 1, dt=0.02, Lrange=(1, 40), L0=20, target_ratio=0.65, seed=991206,
                                    nsamples=ntraj - ntraj // 2, ndraws=ntraj // 2, max_iters=ntraj)
        # the reference's uncapped L = max(1, int(lambda/dt)) (hmcda.py:307), bounded by wall clock
        ctx.set_hmc_options(0, args.da_budget)
        legs["da_uncapped"] = run_leg(B * world, 1, dt=0.02, Lrange=(1, 0), L0=20, target_ratio=0.65, seed=991206,
                                      nsamples=ntraj - ntraj // 2, ndraws=ntraj // 2, max_iters=ntraj)
        ctx.set_hmc_options(0, 0.0)
        ctx.config_obs(dobs)
        hmc = legs

    # ---- max / sum over ranks
    tt = torch.tensor([ms, t_e2e * 1e3] + ([strong[0]] if strong else []), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(tt[0]), float(tt[1])
    hmc_out = None
    if hmc is not None:
        hmc_out = {}
        for name, L in hmc.items():
            vmax = torch.tensor([L["t"], L["t_gather"], L["t_wait"]], dtype=torch.float64, device=dev)
            vsum = torch.tensor([L["evals"]], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(vmax, op=dist.ReduceOp.MAX)
                dist.all_reduce(vsum, op=dist.ReduceOp.SUM)
            t = float(vmax[0])
            hmc_out[name] = {"chains_total": L["chains"], "seconds": t, "trajectories_per_s": L["traj"] / t,
                             "accepted_samples_per_s": L["acc"] / t, "evals_per_s": float(vsum[0]) / t,
                             "global_steps_rank0": L["steps"],
                             "nccl_gather_ms": 1e3 * float(vmax[1]), "rank_imbalance_wait_ms": 1e3 * float(vmax[2]),
                             "gathered_misfit_shape": L["misfit_shape"]}
        desc = {"c4_strong": "HamitonianMC, L=20, dt=0.02, 16 384 chains in total sharded over the GPUs (strong "
                             "scaling), %d trajectories per chain; includes chain initialisation, the NCCL "
                             "broadcast of the observations and the all-gathers of misfit / counters" % args.hmc_traj,
                "base_weak": "HamitonianMC, L=20, dt=0.02, %d chains per GPU, 10 trajectories each" % B,
                "da_capped": "HMCDualAveraging, L0=20, dt0=0.02, target 0.65, L capped at 40 (extension), %d "
                             "chains per GPU, %d trajectories each (first half adapts the step size; includes "
                             "_find_initial_dt)" % (B, args.hmc_traj),
                "da_uncapped": "HMCDualAveraging as the reference: L = max(1, int(lambda/dt)) uncapped "
                               "(hmcda.py:307), same settings, stopped after %.0f s of wall clock (a warm-up "
                               "rejection sends L to ~4e5 for that chain)" % args.da_budget}
        for k in hmc_out:
            hmc_out[k]["sampler"] = desc[k]
    value = world * B * args.steps / (ms * 1e-3)
    e2e_val = world * B * args.steps / (ms_e2e * 1e-3)

    out = None
    if rank == 0:
        hbm_peak = 6558.7
        try:
            hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        except Exception:
            pass
        # ---- rooflines from the live per-kernel times
        evals_per_launch = nev / max(1, args.steps)
        nsolve = 3 * 36            # sequences T, 1.05 T, 0.95 T x 36 periods (Rc and Rg share the T sequence)
        n2 = 65
        work = {"swd_roots": evals_per_launch * (N_LAYERS - 1) * F_R,
                "swd_eigen": B * nsolve * N_LAYERS * E_R,
                "rf_propagate": B * n2 * N_LAYERS * P_RF}
        tot_ms = sum(kms.values())
        kernels = {}
        for k, v in kms.items():
            if klaunch[k] == 0:
                continue
            e = {"ms": round(v, 4), "launches": klaunch[k], "share_of_step": round(v / tot_ms, 4)}
            if k in work:
                e["tflops"] = work[k] / (v * 1e-3) / 1e12
                e["fp64_frac"] = e["tflops"] / fp64_peak if fp64_peak else None
            kernels[k] = e
        by_spec = B * (2 * n2 + 2 * N_LAYERS * n2) * 16.0
        if "rf_propagate" in kernels:
            kernels["rf_propagate"]["hbm_gbs"] = by_spec / (kms["rf_propagate"] * 1e-3) / 1e9
        if "rf_decon" in kernels:
            by = by_spec + B * (125 + 1 + 2 * N_LAYERS) * 8.0
            kernels["rf_decon"]["hbm_gbs"] = by / (kms["rf_decon"] * 1e-3) / 1e9
            kernels["rf_decon"]["hbm_frac"] = kernels["rf_decon"]["hbm_gbs"] / hbm_peak
        k1 = kernels.get("swd_roots", {})
        roofline = {"bound": "fp64", "kernel": "swd_roots_kernel", "achieved": k1.get("tflops"),
                    "peak": fp64_peak, "unit": "TFLOP/s", "frac": k1.get("fp64_frac"), "traffic": None,
                    "kernel_ms": kms.get("swd_roots"), "share_of_step": k1.get("share_of_step"),
                    "note": "all measured in this run: peak = DFMA micro-benchmark (MEASURED_PEAKS.json has no "
                            "FP64 figure); achieved = secular evaluations counted on device x (n-1) layer steps x "
                            "F_R=375 flop / kernel time from CUDA events around the launch (median of 5 "
                            "rfs_profile_eval calls, RF branch serialised so that the kernel runs alone); "
                            "kernel_ms is the whole root-search stage: the search kernel plus the two small "
                            "kernels that build the length-sorted job order, whose 7 evaluations per job are "
                            "NOT counted as algorithmic work",
                    "secular_evals_per_launch": evals_per_launch,
                    "root_search_mapping": {"T": mapping_main[0], "S": mapping_main[1],
                                            "length_sorted_job_order": bool(sorted_main)}}
        for fn in ("r02_traffic.json", "r01_traffic.json"):
            tr = os.path.join(ROOT, "profiles", fn)
            if os.path.exists(tr):
                try:
                    roofline["traffic"] = json.load(open(tr)).get("swd_roots_kernel_dram_bytes_per_launch")
                    roofline["traffic_source"] = "profiles/" + fn + " (ncu --set full; not on the value path)"
                    break
                except Exception:
                    pass
        cpu = None
        if not args.no_cpu_baseline:
            cfg2, _, Xc = workload(4096, 4321)
            v, done, dtc = cpu_arm(cfg2, dobs, Xc, args.cpu_seconds, ncores)
            cpu = {"value": v, "unit": "evals/s", "cores": ncores, "kind": "port",
                   "sample": "%d evaluations of the same workload in %.1f s (oracle restatement, g++ -O3, "
                             "%d threads)" % (done, dtc, ncores)}
        configs = None
        if world == 1 and not args.no_configs:
            configs = config_legs(torch, local_rank, ncores, hbm_peak, fp64_peak, with_cpu=not args.no_cpu_baseline)
        out = {"metric": "joint RF+SWD forward+gradient evaluations/s", "value": value, "unit": "evals/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic", "config": config, "clocks": sampler.summary(),
               "e2e": {"value": e2e_val, "unit": "evals/s", "h2d_bytes_per_step": B * 2 * N_LAYERS * 8,
                       "d2h_bytes_per_step": B * (1 + 2 * N_LAYERS + nd) * 8 + B, "gpu_launches": launches_e2e,
                       "api": "rfsurfhmc_b200.batched.HostPipeline (2 slots: copies overlap the next batch)"},
               "gpu_launches": launches, "roofline": roofline, "kernels": kernels,
               "kernels_note": "ms / share: CUDA events around every launch in this run.  tflops = algorithmic "
                               "flop by the frozen hand counts of BASELINE.md §3 (1 FMA = 2, div/sqrt/exp/sin/cos "
                               "= 20 flop each; E_R and P_RF are generous per-layer counts) / kernel time; the FP64 "
                               "pipe utilisation ncu measures for the same kernels is in profiles/r02_kernels.md "
                               "(roots 58 %, eigen 54 %, RF propagate 66 %)",
               "cpu_baseline": cpu,
               "hmc": hmc_out, "configs": configs, "failed_models_last_step": n_fail}
        if strong is not None:
            ms_s = float(tt[2])
            out["strong_scaling"] = {"chains_total": strong[1] * world, "chains_per_gpu": strong[1],
                                     "value": world * strong[1] * args.steps / (ms_s * 1e-3), "unit": "evals/s",
                                     "ms_per_step": ms_s / args.steps,
                                     "root_search_mapping": {"T": strong[2][0], "S": strong[2][1]},
                                     "note": "BASELINE config 4: 16 384 chains in total sharded over the GPUs; "
                                             "compare with `value` of the N=1 run"}
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
