"""Drivers with the behaviour of /root/reference/main_base.py:14-93 and main_DA.py:12-91:
read param.yaml, synthesise observations from `true_model`, build the search box, run the chains,
write `real_syn.npy`, per-chain result files and `misfit.npy [nchains, nsamples]`.

    python -m rfsurfhmc_b200.driver --param param.yaml --sampler base --chains 4
    torchrun --nproc-per-node 8 -m rfsurfhmc_b200.driver --sampler da --chains 16384

`mpiexec -n N` of the reference becomes `--chains N`: all chains of a rank run at once on its GPU.
In the parameter file, rf.ray_p may be a list of ray parameters and rf.gauss a list of Gaussian widths
(e.g. `gauss: [1.0, 2.5]`): the receiver-function data are then one trace per (ray, width), in that order.
An optional `true_model.vpvs: [n values]` samples each layer's Vp/Vs ratio as a third parameter block:
models are [vs, thk, vpvs] (vp = vpvs * vs, density from Brocher's polynomial of vp), the observations are
synthesised from [vs, thk, vpvs] and the Vp/Vs box is +-10 % of the true values (fixtures.driver_bounds_vpvs).

    python -m rfsurfhmc_b200.driver --param param.yaml --stations stations.npz --chains K

inverts a station array instead: the observations of S stations come from the file (see
model/stations.py: load_stations; the optional key ray_p [S] or [S, nray] gives each station its own
ray parameter(s) in place of rf.ray_p, swd_use [S, nper] the periods of the swd lists it observes,
rf_use [S, nray*ngauss*nt] or [S, nray, ngauss, nt] ([S, nray, nt] with one width) the
receiver-function samples it fits: missing ray bins, fitting windows, and gauss [S] or [S, ngauss] its
own Gaussian width(s) in place of rf.gauss: the widths its data were processed with), K chains run per station, all S*K in one device run (sharded
over ranks under torchrun), and {outdir}/{name}/misfit.npy [K, nsamples] is written per station.  With
true_model.vpvs the file's bounds are [S, 3n, 2]."""
import argparse
import os
import time
import numpy as np
import yaml

from .model.model_rf import ReceiverFunc
from .model.model_surf import SurfWD
from .model.model_rf_swd_vs_thk import Joint_RF_SWD
from .model.stations import StationArray, load_stations
from .pyhmc.hmc import HamitonianMC
from .pyhmc.hmcda import HMCDualAveraging
from .fixtures import driver_bounds, driver_bounds_vpvs
from . import distributed as D


def run(param, sampler="base", nchains=4, save_chains=True, max_iters=0, max_L=0, stations=None):
    """stations: None (observations synthesised from `true_model`, as the reference) or a stations file
    / mapping (load_stations): then `nchains` chains run per station."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if ws > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    vpvs = param['true_model'].get('vpvs')
    model_swd = SurfWD.init(**param['swd'], vpvs=vpvs is not None)
    model_rf = ReceiverFunc.init(**param['rf'], vpvs=vpvs is not None)
    thk = np.asarray(param['true_model']['thk'], dtype=np.float64)
    vs = np.asarray(param['true_model']['vs'], dtype=np.float64)
    model_swd.set_thk(thk)
    model_rf.set_thk(thk)
    model = Joint_RF_SWD(1.0, 1.0, model_rf, model_swd)
    model.set_device(local)
    outdir = param['hmc']['OUTPUT_DIR']
    os.makedirs(outdir, exist_ok=True)
    x = np.hstack((vs, thk))
    bounds_of = driver_bounds
    if vpvs is not None:
        k = np.asarray(vpvs, dtype=np.float64)
        if k.shape != vs.shape:
            raise ValueError(f"true_model.vpvs has {k.size} values for {vs.size} layers")
        x = np.hstack((vs, thk, k))
        bounds_of = driver_bounds_vpvs
    if stations is None:
        dobs = np.zeros(model.ndata)
        if rank == 0:
            drsyn, dssyn, _ = model.forward(x)
            dobs[:model.rfmodel.nt] = drsyn
            dobs[model.rfmodel.nt:] = dssyn
            np.save(f"{outdir}/real_syn.npy", dobs)
        dobs = D.bcast_array(dobs)
        nt = model.rfmodel.nt
        model.set_obsdata(dobs[:nt], dobs[nt:])
        boundaries = bounds_of(x)
        npairs = nchains
        ids, sidx = D.shard_chains(nchains), None
    else:
        st = load_stations(stations, model.ndata, x.size, bounds_of(x), model_rf.nray, model_swd, model_rf,
                           model_rf.ngauss)
        model = StationArray(model, st["dobs"], st["sigma1"], st["sigma2"], st["names"], st["ray_p"],
                             st["swd_use"], st["rf_use"], st["gauss"])
        boundaries = st["bounds"]
        npairs = model.nstations * nchains
        sidx, ids = D.shard_station_chains(model.nstations, nchains)
    cls = HamitonianMC if sampler == "base" else HMCDualAveraging
    chain = cls.init(model, boundaries, 0, **param['hmc'])
    chain.max_iters = int(max_iters)  # 0 = unbounded, as the reference's `while True` loops
    if sampler == "da":
        chain.max_L = int(max_L)      # 0 = the reference's uncapped L = int(lambda/dt)
    if npairs < ws:
        raise ValueError("need at least one chain per rank (chains %d < world size %d)" % (npairs, ws))
    if save_chains:
        # per-chain files need every accepted sample's synthetics on the host: [chains, nsamples, ndata];
        # the decision is collective (max over ranks) so that no rank leaves the others in a gather
        need = D.max_over_ranks(len(ids) * float(param['hmc']['nsamples']) * model.ndata * 8)
        if need > 8e9:
            raise MemoryError("per-chain result files for %d chains need %.1f GB of synthetics per rank; "
                              "run with --no-chain-files (misfit.npy is still written)" % (len(ids), need / 1e9))
    out = chain.sample_chains(ids, want_syn=save_chains, save=save_chains, stations=sidx)
    # end-of-run gathers (replace comm.Gather at main_base.py:90): misfit history + per-chain counters
    t0 = time.perf_counter()
    misfit = D.gather_chains(out["misfit"], npairs)
    n_iter = D.gather_chains(out["n_iter"], npairs)
    n_acc = D.gather_chains(out["n_acc"], npairs)
    complete = D.gather_chains(out["complete"].astype(np.int64), npairs).astype(bool)
    out["gather_ms"] = 1e3 * (time.perf_counter() - t0)
    out["n_acc_all"], out["complete_all"] = n_acc, complete
    if rank == 0:
        # rows an incomplete chain never filled are NaN (never 0.0: argsort would pick them as "best")
        if sidx is None:
            np.save(f"{outdir}/misfit.npy", misfit)
        else:
            for s, name in enumerate(model.names):
                os.makedirs(f"{outdir}/{name}", exist_ok=True)
                np.save(f"{outdir}/{name}/misfit.npy", misfit[s * nchains:(s + 1) * nchains])
    return misfit, n_iter, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--param", default="param.yaml")
    ap.add_argument("--sampler", default="base", choices=["base", "da"])
    ap.add_argument("--chains", type=int, default=4, help="chains (per station with --stations)")
    ap.add_argument("--stations", default=None,
                    help="stations .npz (dobs [S,ndata]; optional names, sigma1, sigma2 [S], bounds [S,2n,2] "
                         "([S,3n,2] with true_model.vpvs), "
                         "ray_p [S] or [S,nray] in place of rf.ray_p, swd_use [S,nper] observed periods of the "
                         "swd lists, rf_use [S,nray*ngauss*nt] or [S,nray,ngauss,nt] fitted RF samples, gauss [S] or "
                         "[S,ngauss] in place of rf.gauss): invert every "
                         "station "
                         "instead of "
                         "observations synthesised from true_model")
    ap.add_argument("--no-chain-files", action="store_true")
    ap.add_argument("--outdir", default=None, help="override hmc.OUTPUT_DIR of the parameter file")
    ap.add_argument("--nsamples", type=int, default=None, help="override hmc.nsamples")
    ap.add_argument("--ndraws", type=int, default=None, help="override hmc.ndraws")
    ap.add_argument("--max-iters", type=int, default=0,
                    help="stop a chain after this many trajectories (0 = unbounded, as the reference)")
    ap.add_argument("--max-L", type=int, default=0,
                    help="dual averaging only: cap on leapfrog steps per trajectory (0 = uncapped)")
    a = ap.parse_args()
    with open(a.param, "r") as f:
        param = yaml.safe_load(f)
    for key, val in (("OUTPUT_DIR", a.outdir), ("nsamples", a.nsamples), ("ndraws", a.ndraws)):
        if val is not None:
            param['hmc'][key] = val
    tic = time.time()
    misfit, n_iter, out = run(param, a.sampler, a.chains, not a.no_chain_files, a.max_iters, a.max_L,
                              a.stations)
    if int(os.environ.get("RANK", "0")) == 0:
        comp = out["complete_all"]
        print("chains %d (%d complete), kept samples %d, accept ratio %.3f" %
              (misfit.shape[0], int(comp.sum()), int(np.isfinite(misfit).sum()),
               out["n_acc_all"].sum() / max(1, n_iter.sum())))
        if not comp.all():
            print("WARNING: %d chain(s) stopped early (max-iters or a failing state): their unfilled rows "
                  "in misfit.npy are NaN and their chain files are flagged complete=False"
                  % int((~comp).sum()))
        print("time elapse: {}".format(time.time() - tic))
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
