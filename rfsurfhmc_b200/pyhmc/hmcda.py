"""HMCDualAveraging — front end with the constructor / `init` / `sample` surface of
/root/reference/pyhmc/hmcda.py (class HMCDualAveraging :11-399), backed by the device-resident
sampler (rfs_hmc_run, sampler=1): `_find_initial_dt`, L = max(1, int(lambda/dt)), always-drawn u and
the Hoffman-Gelman dual-averaging recursion run per chain on the GPU (hmc_kernels.cuh)."""
import numpy as np
from ._common import require_device_model, finish_run, save_chains, station_run_args


class HMCDualAveraging:
    def __init__(self, UserDefinedModel, boundaries, dt: float, L0: int, nbest_model: int,
                 target_ratio: float, seed: int, nsamples: int, ndraws: int, myrank=0, name="mychain",
                 outdir="./"):
        self.model = require_device_model(UserDefinedModel)
        self.boundaries = np.asarray(boundaries, dtype=np.float64)
        self.dt = dt
        self.L = L0
        self.nbest_model = nbest_model
        self.nsamples = nsamples
        self.ndraws = ndraws
        if ndraws < 0.1 * nsamples:
            raise ValueError(f"in dual averaging, ndraws should > nsamples * 0.1 "
                             f"(ndraws = {ndraws}, nsamples = {nsamples})")  # reference: exit(1), hmcda.py:55-58
        self.seed = seed + myrank
        self._base_seed = seed
        self.myrank = myrank
        self.name = name
        self.outdir = outdir
        self.delta = target_ratio
        self.max_iters = 0
        self.max_L = 0   # extension: cap on L = max(1, int(lambda/dt)); 0 = unlimited (reference)
        self.last = None

    @classmethod
    def init(self, UserDefinedModel, boundaries, rank, **kargs):
        return HMCDualAveraging(UserDefinedModel, boundaries, kargs['dt'], kargs['L0'], kargs['nbest'],
                                kargs['target_ratio'], kargs['seed'], kargs['nsamples'], kargs['ndraws'],
                                rank, kargs['name'], kargs['OUTPUT_DIR'])

    def sample_chains(self, chain_ids, want_syn=True, log_accepts=0, save=False, stations=None):
        n, sets = station_run_args(self.model, self.boundaries, chain_ids, stations)
        ctx = self.model.device_context(n)
        out = ctx.hmc_run(1, chain_ids, self.boundaries, self.dt, Lrange=(1, self.max_L), L0=self.L,
                          target_ratio=self.delta,
                          seed=self._base_seed, nsamples=self.nsamples, ndraws=self.ndraws,
                          max_iters=self.max_iters, want_samples=True, want_syn=want_syn,
                          log_accepts=log_accepts, which=self.model.which, sets=sets)
        finish_run(out, self.nsamples, self.ndraws)
        out["station"] = sets
        if save:
            # nbests hard-coded to 10 in the reference (hmcda.py:359)
            save_chains(self.model, out, chain_ids, sets, self.outdir, self.name, 10, self.nsamples)
        self.last = out
        return out

    def sample(self):
        out = self.sample_chains([self.myrank], want_syn=True, save=True)
        return out["misfit"][0]
