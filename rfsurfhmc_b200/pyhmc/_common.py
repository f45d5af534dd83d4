"""Shared pieces of the two sampler front ends: result files and the device-run wrapper."""
import os
import numpy as np


def finish_run(out, nsamples, ndraws):
    """Post-process a Context.hmc_run result: rows a chain never filled (stopped by max_iters, stuck at
    a failing state, failure in _find_initial_dt) become NaN instead of 0.0, `n_valid` / `complete`
    are added, and the library's warning is surfaced."""
    import warnings
    nvalid, complete = chain_status(out, nsamples, ndraws)
    out["n_valid"], out["complete"] = nvalid, complete
    for i in np.nonzero(~complete)[0]:
        out["misfit"][i, nvalid[i]:] = np.nan
        if out.get("samples") is not None:
            out["samples"][i, nvalid[i]:] = np.nan
        if out.get("syn") is not None:
            out["syn"][i, nvalid[i]:] = np.nan
    if out.get("warning"):
        warnings.warn(out["warning"], RuntimeWarning)
    if not complete.all():
        warnings.warn("%d of %d chain(s) stopped before nsamples accepted samples (max_iters or a failing "
                      "state); their unfilled rows are NaN" % (int((~complete).sum()), complete.size),
                      RuntimeWarning)
    return out


def station_run_args(model, boundaries, chain_ids, stations):
    """(n, sets) for Context.hmc_run: the layer count from `boundaries` ([P n,2] or [S,P n,2], P = 3 for
    a model with vpvs=True, else 2) and the station of each chain (None without a StationArray).  Chain i
    samples station stations[i]."""
    from ..model import param
    b = np.asarray(boundaries)
    if b.ndim not in (2, 3) or b.shape[-1] != 2:
        raise ValueError(f"boundaries must be [2n, 2] or [S, 2n, 2], got shape {b.shape}")
    vpvs = bool(getattr(model, "vpvs", False))
    n = param.layer_count(b.shape[-2], vpvs)
    param.check_vpvs_box(b, vpvs)
    if stations is None:
        return n, None
    if not hasattr(model, "station_model"):
        raise ValueError("stations= needs a StationArray model")
    st = np.asarray(stations, dtype=np.int64)
    if st.shape != np.shape(np.atleast_1d(chain_ids)):
        raise ValueError("stations must give one station per chain id")
    if b.ndim == 3 and b.shape[0] != model.nstations:
        raise ValueError(f"boundaries has {b.shape[0]} boxes for {model.nstations} stations")
    return n, st


def save_chains(model, out, chain_ids, stations, outdir, name, nbest, nsamples):
    """Write every chain of a run: {outdir}/{name}.{cid}.npz, or {outdir}/{station name}/{name}.{cid}.npz
    with the station's observations and synthetics when the chains sample a StationArray."""
    single = {}
    for i, cid in enumerate(np.atleast_1d(chain_ids)):
        if stations is None:
            save_chain(f"{outdir}/{name}.{int(cid)}.npz", model, out, i, nbest, nsamples)
            continue
        s = int(stations[i])
        if s not in single:
            # with per-station periods or RF samples the file keeps the array's data layout, as the chain's
            # syn rows do
            masked = model.swd_use is not None or model.rf_use is not None
            single[s] = model.station_view(s) if masked else model.station_model(s)
        save_chain(f"{outdir}/{model.names[s]}/{name}.{int(cid)}.npz", single[s], out, i, nbest, nsamples)


def save_chain(path, model, out, i, nbest, nsamples):
    """Write chain i of a device run.  Only the rows the chain really produced are stored; incomplete
    chains are flagged (`complete` = False)."""
    nv = int(out["n_valid"][i])
    xmean = best_mean_model(out["misfit"][i], out["samples"][i], nbest, nv)
    dsyn = np.full(np.asarray(model.dobs).shape, np.nan)
    if np.all(np.isfinite(xmean)):
        dsyn = model.misfit_and_grad(xmean)[2]
    syn = out["syn"][i][:nv] if out["syn"] is not None else np.zeros((nv, 0))
    write_chain_file(path, out["initmodel"][i], model.dobs, xmean, dsyn, out["samples"][i][:nv], syn,
                     complete=bool(out["complete"][i]))


def write_chain_file(path, initmodel, obs, xmean, synmean, samples, syn, complete=True):
    """Per-chain result file with the logical layout of the reference's HDF5 output
    (/root/reference/pyhmc/hmc.py:203-226,272-275): datasets `initmodel`, `obs`, groups
    `mean/{model,syn}` and `{i}/{model,syn}`.  h5py is not available in this image, so the same
    tree is stored in an .npz: keys "initmodel", "obs", "mean/model", "mean/syn", "models"
    ([nsamples,2n] == {i}/model stacked) and "syn" ([nsamples,ndata] == {i}/syn stacked).
    `tools/npz_to_h5.py` converts to the reference's exact HDF5 tree where h5py exists."""
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    np.savez(path, **{"initmodel": initmodel, "obs": obs, "mean/model": xmean, "mean/syn": synmean,
                      "models": samples, "syn": syn, "complete": np.bool_(complete)})


def best_mean_model(misfit, samples, nbest, nvalid=None):
    """Average of the nbest lowest-misfit samples (hmc.py:266-270).  nvalid: number of rows that were
    really filled (a chain stopped by max_iters / a failing state has fewer than nsamples)."""
    if nvalid is not None:
        misfit, samples = misfit[:nvalid], samples[:nvalid]
    if misfit.shape[0] == 0:
        return np.full(samples.shape[1], np.nan)
    idx = np.argsort(misfit)
    return np.mean(samples[idx[:nbest], :], axis=0)


def require_device_model(model):
    """The reference samplers accept any object with misfit_and_grad (pyhmc/hmc.py:113-119) and call
    it from a Python loop.  Here the loop itself runs on the GPU, so the model must be one of the
    three device-backed objectives (Joint_RF_SWD, ReceiverFunc, SurfWD: `device_context(n)` +
    `which`); an arbitrary Python callable cannot be sampled -- there is no CPU/Python fallback."""
    if not (hasattr(model, "device_context") and hasattr(model, "which")):
        raise TypeError(
            "rfsurfhmc_b200 samplers run the chains on the GPU and need a device-backed model "
            "(rfsurfhmc_b200.model: Joint_RF_SWD, ReceiverFunc or SurfWD); arbitrary Python "
            "models are not supported: there is no CPU/Python fallback loop")
    return model


def chain_status(out, nsamples, ndraws):
    """Per-chain completion of a device run: (n_valid_samples [C], complete [C] bool)."""
    nvalid = np.clip(np.asarray(out["n_acc"]) - ndraws, 0, nsamples)
    return nvalid, nvalid >= nsamples
