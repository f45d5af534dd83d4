"""Batched device API: torch tensors in, torch tensors out (PyTorch only hands over device memory
and the current stream; all numerics are in librfsurf_b200.so)."""
import torch
from ._lib import Context


class JointEvaluator:
    """Many-chains Joint_RF_SWD.misfit_and_grad on one GPU with resident inputs/outputs.  dobs [ndata]
    or [S, ndata]: S observation sets (stations) sharing `cfg`; cfg's sigma1 / sigma2 may then be
    [S] arrays.  cfg's gauss may be a list of Gaussian widths: the RF block of the data vector is then
    [ray][gauss][nt].  obs_ray_p [S] or [S, nray]: each set's own ray parameter(s) in place of cfg's
    ray_p (for every width).  obs_swd_use [S, nper]: the periods of cfg's lists (the common grid) each set
    observes.  obs_rf_use [S, nray * ngauss * nt], [S, nray, ngauss, nt] or [S, nray, nt]: the
    receiver-function samples each set fits.  obs_gauss [S] or [S, ngauss]: each set's own Gaussian
    width(s) in place of cfg's gauss (for every ray)."""

    def __init__(self, cfg, dobs, nlayer, device=0, which=0, obs_ray_p=None, obs_swd_use=None, obs_rf_use=None,
                 obs_gauss=None):
        self.ctx = Context(device)
        self.which = which
        self.n = nlayer
        if which != 1:
            self.ctx.config_swd(nlayer, cfg.get("tRc"), cfg.get("tRg"), cfg.get("tLc"), cfg.get("tLg"),
                                mode=cfg.get("mode", 0), sphere=cfg.get("sphere", False),
                                stale=cfg.get("stale", True))
        if which != 2:
            self.ctx.config_rf(nlayer, cfg["ray_p"], cfg["nt"], cfg["dt"], cfg["gauss"], cfg["time_shift"],
                               cfg.get("water", 0.001), cfg.get("rf_type", "P"), cfg.get("method", "freq"))
        self.ctx.config_obs(dobs, cfg.get("sigma1", 1.0), cfg.get("sigma2", 1.0))
        if obs_ray_p is not None:
            self.ctx.config_obs_rays(obs_ray_p)
        if obs_swd_use is not None:
            self.ctx.config_obs_periods(obs_swd_use)
        if obs_rf_use is not None:
            self.ctx.config_obs_rf_samples(obs_rf_use)
        if obs_gauss is not None:
            self.ctx.config_obs_gauss(obs_gauss)
        self.device = torch.device("cuda", device)
        self.ndata = self.ctx.ndata(which)
        self._out = None

    def __call__(self, x, sets=None):
        """x: float64 CUDA tensor [B, 2n] -> (U [B], grad [B,2n], dsyn [B,ndata], flag [B] uint8).
        sets: int32 CUDA tensor [B], the observation set of each row (required with several sets)."""
        assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous()
        B = x.shape[0]
        if sets is not None:
            assert sets.is_cuda and sets.dtype == torch.int32 and sets.is_contiguous() and sets.shape == (B,)
        if self._out is None or self._out[0].shape[0] != B:
            self._out = (torch.empty(B, dtype=torch.float64, device=self.device),
                         torch.empty(B, 2 * self.n, dtype=torch.float64, device=self.device),
                         torch.empty(B, self.ndata, dtype=torch.float64, device=self.device),
                         torch.empty(B, dtype=torch.uint8, device=self.device))
        U, G, D, F = self._out
        self.ctx.misfit_grad_dev(B, x.data_ptr(), self.which, U.data_ptr(), G.data_ptr(), D.data_ptr(),
                                 F.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream,
                                 sets.data_ptr() if sets is not None else 0)
        return U, G, D, F


class HostPipeline:
    """Host-buffer front end for streams of independent batches (the end-to-end path of bench.py):
    `submit(x_host)` copies the batch from pinned host memory, evaluates it and copies U, grad,
    dsyn, flag back to pinned host buffers, double-buffered over two slots (own context, stream and
    buffers each) so that the copies of one batch overlap the kernels of the next.
    `submit` returns the slot whose previous results are now complete (or None)."""

    def __init__(self, cfg, dobs, nlayer, batch, device=0, which=0, slots=2):
        self.dev = torch.device("cuda", device)
        self.B, self.n, self.which = batch, nlayer, which
        self.slots = []
        for _ in range(slots):
            ev = JointEvaluator(cfg, dobs, nlayer, device, which)
            nd = ev.ndata
            slot = {
                "ev": ev, "stream": torch.cuda.Stream(self.dev), "event": torch.cuda.Event(), "busy": False,
                "x": torch.empty(batch, 2 * nlayer, dtype=torch.float64, device=self.dev),
                "U": torch.empty(batch, dtype=torch.float64, device=self.dev),
                "G": torch.empty(batch, 2 * nlayer, dtype=torch.float64, device=self.dev),
                "D": torch.empty(batch, nd, dtype=torch.float64, device=self.dev),
                "F": torch.empty(batch, dtype=torch.uint8, device=self.dev),
                "Uh": torch.empty(batch, dtype=torch.float64).pin_memory(),
                "Gh": torch.empty(batch, 2 * nlayer, dtype=torch.float64).pin_memory(),
                "Dh": torch.empty(batch, nd, dtype=torch.float64).pin_memory(),
                "Fh": torch.empty(batch, dtype=torch.uint8).pin_memory(),
            }
            self.slots.append(slot)
        self.i = 0
        self.h2d_bytes = batch * 2 * nlayer * 8
        self.d2h_bytes = batch * (1 + 2 * nlayer + self.slots[0]["D"].shape[1]) * 8 + batch

    @property
    def launches(self):
        return sum(s["ev"].ctx.launches for s in self.slots)

    def submit(self, x_host):
        """x_host: pinned float64 [B, 2n].  Returns the completed previous result of the slot that
        is being reused as (U, grad, dsyn, flag) pinned host tensors, or None."""
        s = self.slots[self.i % len(self.slots)]
        self.i += 1
        done = None
        if s["busy"]:
            s["event"].synchronize()
            done = (s["Uh"], s["Gh"], s["Dh"], s["Fh"])
        with torch.cuda.stream(s["stream"]):
            s["x"].copy_(x_host, non_blocking=True)
            s["ev"].ctx.misfit_grad_dev(self.B, s["x"].data_ptr(), self.which, s["U"].data_ptr(),
                                        s["G"].data_ptr(), s["D"].data_ptr(), s["F"].data_ptr(),
                                        s["stream"].cuda_stream)
            s["Uh"].copy_(s["U"], non_blocking=True)
            s["Gh"].copy_(s["G"], non_blocking=True)
            s["Dh"].copy_(s["D"], non_blocking=True)
            s["Fh"].copy_(s["F"], non_blocking=True)
            s["event"].record(s["stream"])
        s["busy"] = True
        return done

    def drain(self):
        """Wait for everything in flight; returns the results of the last submitted batch."""
        last = None
        for k in range(len(self.slots)):
            s = self.slots[(self.i + k) % len(self.slots)]
            if s["busy"]:
                s["event"].synchronize()
                s["busy"] = False
                last = (s["Uh"], s["Gh"], s["Dh"], s["Fh"])
        return last
