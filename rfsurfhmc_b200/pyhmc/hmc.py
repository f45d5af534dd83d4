"""HamitonianMC — front end with the constructor / `init` / `sample` surface of
/root/reference/pyhmc/hmc.py (class HamitonianMC :9-276), backed by the device-resident sampler
(include/rfsurfhmc.h: rfs_hmc_run, sampler=0).

The leapfrog loop, reflections, Metropolis step and the NumPy-legacy random stream all live in
hmc_kernels.cuh; chain `myrank` is seeded with `seed + myrank` exactly like one MPI rank of the
reference (hmc.py:43,61), so `sample()` reproduces that rank's accept/reject sequence, and
`sample_chains(ids)` runs any number of ranks at once on one GPU."""
import numpy as np
from ._common import require_device_model, finish_run, save_chains, station_run_args


class HamitonianMC:
    def __init__(self, UserDefinedModel, boundaries, dt, Lrange, nbest_model, seed, nsamples, ndraws,
                 myrank=0, name="mychain", outdir="./"):
        self.myrank = myrank
        self.seed = seed + myrank
        self._base_seed = seed
        self.boundaries = np.asarray(boundaries, dtype=np.float64)
        self.Lrange = Lrange
        self.dt = dt
        self.model = require_device_model(UserDefinedModel)
        self.nbest_model = nbest_model
        self.nsamples = nsamples
        self.ndraws = ndraws
        self.name = name
        self.outdir = outdir
        self.max_iters = 0
        self.last = None

    @classmethod
    def init(self, UserDefinedModel, boundaries, rank, **kargs):
        return HamitonianMC(UserDefinedModel, boundaries, kargs['dt'], kargs['Lrange'], kargs['nbest'],
                            kargs['seed'], kargs['nsamples'], kargs['ndraws'], rank, kargs['name'],
                            kargs['OUTPUT_DIR'])

    def sample_chains(self, chain_ids, want_syn=True, log_accepts=0, save=False, stations=None):
        """Run the chains `chain_ids` (the reference's MPI ranks) at once; returns the result dict of
        Context.hmc_run (misfit [C,nsamples], samples, syn, initmodel, n_iter, n_acc, ...)."""
        n, sets = station_run_args(self.model, self.boundaries, chain_ids, stations)
        ctx = self.model.device_context(n)
        out = ctx.hmc_run(0, chain_ids, self.boundaries, self.dt, Lrange=self.Lrange, seed=self._base_seed,
                          nsamples=self.nsamples, ndraws=self.ndraws, max_iters=self.max_iters,
                          want_samples=True, want_syn=want_syn, log_accepts=log_accepts,
                          which=self.model.which, sets=sets)
        finish_run(out, self.nsamples, self.ndraws)
        out["station"] = sets
        if save:
            save_chains(self.model, out, chain_ids, sets, self.outdir, self.name, self.nbest_model, self.nsamples)
        self.last = out
        return out

    def sample(self):
        """One chain (this rank), as the reference: returns misfit[nsamples] and writes
        {outdir}/{name}.{myrank}.npz."""
        out = self.sample_chains([self.myrank], want_syn=True, save=True)
        return out["misfit"][0]
