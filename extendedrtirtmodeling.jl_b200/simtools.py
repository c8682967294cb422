"""Host-side mirror of the reference's simulation-study layer around the sweep path (src/SimTools.jl:385-553):
checkConvergence, runSimulation, getMetrics, getMetrics2, comparePara.  These are the callers either side of the hot
path (SURVEY.md 8f-2, 8f-3): runSimulation draws nRep data sets from one set of true parameters, fits each with the
GPU sampler and keeps posterior means, DIC and the convergence summary, in the reference's Dict layout so that
getMetrics* read it unchanged.  Replications are independent, so they shard over GPUs/processes with no collective:
replication r runs on rank r mod world (one process per GPU), results are gathered at the end."""
import numpy as np

from . import api, simulate
from .diagnostics import ess_rhat_batched, ess_rhat_device


def checkConvergence(MCMC, device=None):
    """src/SimTools.jl:419-443: share of the traced columns of Post.ra / Post.rt / Post.qr with ESS > 400 and R-hat < 1.1
    after burn-in (constant columns give NaN and are not counted, as with MCMCChains).  One batched computation per block:
    device="cuda" (or a device index) runs the CUDA kernel of the engine (erirt_ess_rhat, one CTA per column), device=None the
    same estimator in torch on the host (reporting on a machine without a GPU)."""
    nb = MCMC.Cond.nBurnin
    ess_ok = rhat_ok = n_ess = n_rhat = 0
    for name in ("ra", "rt", "qr"):
        arr = getattr(MCMC.Post, name, None)
        if arr is None or arr.size == 0:
            continue
        arr = np.asarray(arr)[nb:]
        keep = np.all(np.isfinite(arr), axis=(0, 2))  # person columns are NaN when person_trace=False
        if not keep.any():
            continue
        if device is None:
            ess, rhat = ess_rhat_batched(arr[:, keep, :], device=None)
        else:
            ess, rhat = ess_rhat_device(arr[:, keep, :], device=0 if device == "cuda" else int(str(device).split(":")[-1]))
        ok = ~np.isnan(ess)
        n_ess += int(ok.sum())
        n_rhat += int((~np.isnan(rhat)).sum())
        ess_ok += int((ess[ok] > 400).sum())
        rhat_ok += int((rhat[~np.isnan(rhat)] < 1.1).sum())
    return dict(ess=100.0 * ess_ok / max(n_ess, 1), rhat=100.0 * rhat_ok / max(n_rhat, 1),
                essN=f"{ess_ok} / {n_ess}", rhatN=f"{rhat_ok} / {n_rhat}")


def _field(P, name):
    return np.asarray(getattr(P, {"σ²t": "sigma2t", "sigma2": "sigma2t"}.get(name, name)))  # InputPara resolves the other Greek aliases


def runSimulation(Cond, truePara, Para=("a", "b", "λ", "σ²t"), funcData=simulate.setDataRtIrt, funcGibbs=api.GibbsRtIrt,
                  typeName="norm", rank=None, world=None, seed=1234, device=None, batch=None, **sample_kwargs):
    """src/SimTools.jl:457-495.  Returns {"True": {p: vector}, 1: {p: posterior mean, "Dic": [DIC], "Diag": {...}}, ..., nRep: {...}}.
    Replication r (1-based) runs on rank (r-1) mod world; with torch.distributed initialised the per-rank results are
    all-gathered so every rank returns the full Dict.  `sample_kwargs` go to api.sample (dtype, person_trace, ...).
    batch=k: each rank runs its replications as replica batches of at most k (api.sampleBatch, one GPU launch sequence per
    batch; not for the Cross family).  A batch keeps no person trace, and the person trace changes the Dict (checkConvergence
    counts the traced theta / zeta columns, and Post.mean.theta feeds D-hat), so batch=k requires person_trace=False and raises
    ValueError otherwise, before any GPU work.  Replication `run` keeps its seeds (sampler seed + run, data seed + run, initial
    values seed + 7919 run), so the Dict is the one batch=None returns with person_trace=False; a batch needs consecutive sampler
    seeds, so with batch the replications are dealt to the ranks in contiguous blocks instead of round robin."""
    if batch is not None:
        if sample_kwargs.get("person_trace", None) is not False:
            raise ValueError("runSimulation(batch=k) keeps no person trace: pass person_trace=False (the sequential run with "
                             "person_trace=False returns the same Dict; its default traces theta / zeta and counts them in Diag)")
        if int(batch) < 1:
            raise ValueError("batch must be a positive number of replications")
    dist = None
    if rank is None or world is None:
        try:
            import torch.distributed as dist_mod
            if dist_mod.is_available() and dist_mod.is_initialized():
                dist = dist_mod
                rank, world = dist.get_rank(), dist.get_world_size()
        except Exception:
            dist = None
        if rank is None or world is None:
            rank, world = 0, 1
    if device is None:
        device = 0
        try:
            import torch
            if torch.cuda.is_available():
                device = rank % max(torch.cuda.device_count(), 1)
        except Exception:
            pass
    Run = {"True": {p: _field(truePara, p).ravel().copy() for p in Para}}
    mine = {}

    def setup(run):
        try:
            Data = funcData(Cond, truePara, type=typeName, rng=seed + run)
        except TypeError:  # generators without error types (setDataRtIrt, setDataRtIrtNull, setDataMlIrt)
            Data = funcData(Cond, truePara, rng=seed + run)
        return funcGibbs(Cond, Data=Data, truePara=truePara, rng=seed + 7919 * run)

    def summary(MCMC, dic):
        Post = {p: _field(MCMC.Post.mean, p).copy() for p in Para}
        Post["Dic"] = [dic]
        Post["Diag"] = checkConvergence(MCMC, device=device)  # ESS / R-hat by the CUDA kernel on the GPU that sampled
        return Post

    dtype = sample_kwargs.get("dtype", "f64")
    if batch is None:
        for run in range(1, Cond.nRep + 1):
            if (run - 1) % world != rank:
                continue
            MCMC = setup(run)
            api.sample(MCMC, seed=seed + run, device=device, **sample_kwargs)
            try:
                dic = api.getDic(MCMC, dtype=dtype, device=device).DIC
            except Exception:  # CrossQr has no D-hat (nu_ij is not traced)
                dic = float("nan")
            mine[run] = summary(MCMC, dic)
    else:
        per = -(-Cond.nRep // world)
        runs = list(range(1 + rank * per, 1 + min(Cond.nRep, (rank + 1) * per)))
        for i in range(0, len(runs), int(batch)):
            group = runs[i:i + int(batch)]
            MCMCs = [setup(run) for run in group]
            api.sampleBatch(MCMCs, seed=seed + group[0], device=device, **sample_kwargs)
            dics = api.getDicBatch(MCMCs, dtype=dtype, device=device)
            for run, MCMC, dic in zip(group, MCMCs, dics):
                mine[run] = summary(MCMC, dic.DIC)
    if dist is not None and world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        for g in gathered:
            Run.update(g)
    else:
        Run.update(mine)
    return Run


def _drop_intercept(est, n_true):
    """vec(β) is column-major over an (nFeat+1) x ncol matrix (ncol = 2 for GibbsRtIrt); the reference's comparePara drops row 1 of
    EVERY column (β[2:end, :], src/SimTools.jl:505), not the first len(est) - len(true) entries of the vector."""
    est = np.asarray(est)
    ncol = est.shape[0] - n_true
    if ncol <= 0 or est.shape[0] % ncol:
        return est
    rows = est.shape[0] // ncol
    m = est.reshape((rows, ncol) + est.shape[1:], order="F")[1:]
    return m.reshape((n_true,) + est.shape[1:], order="F")


def _stack(obj, par):
    runs = sorted(k for k in obj if k != "True")
    true = np.asarray(obj["True"][par], dtype=np.float64).ravel(order="F")  # Julia's vec(): column-major
    est = np.stack([np.asarray(obj[r][par], dtype=np.float64).ravel(order="F") for r in runs], axis=1)
    if par in ("β", "beta"):  # the reference drops the intercept row (src/SimTools.jl:505)
        est = _drop_intercept(est, len(true))
    return true, est


def _mean_corr(est, true):
    cs = [np.corrcoef(est[:, i], true)[0, 1] for i in range(est.shape[1])] if len(true) > 1 else [np.nan]
    return float(np.mean(cs))


def getMetrics(obj, par="a"):
    """src/SimTools.jl:500-524 (over the replications actually present instead of a hard-coded 100)."""
    true, est = _stack(obj, par)
    d = est - true[:, None]
    return dict(Bias=float(d.mean()), Rmse=float(np.sqrt((d ** 2).mean())), Corr=_mean_corr(est, true))


def getMetrics2(obj, par="a"):
    """src/SimTools.jl:528-553."""
    true, est = _stack(obj, par)
    d = est - true[:, None]
    return dict(relativeBias=float((d / true[:, None]).mean()), normalizedRmse=float(np.sqrt((d ** 2).mean()) / (est.max() - est.min())),
                Corr=_mean_corr(est, true))


def comparePara(MCMC, par="a", file=None):
    """src/SimTools.jl:389-414: estimate, truth and absolute difference, rounded to 3 digits."""
    import sys
    out = file or sys.stdout
    true = _field(MCMC.truePara, par).ravel(order="F")  # Julia's vec(): column-major
    est = _field(MCMC.Post.mean, par).ravel(order="F")
    if par in ("β", "beta") and est.shape[0] != true.shape[0]:
        est = _drop_intercept(est, true.shape[0])
    print("Esti\tTrue\t|Diff|", file=out)
    print("=======\t=======\t=======", file=out)
    for e, t in zip(est, true):
        print(f"{round(float(e), 3)}\t{round(float(t), 3)}\t{round(abs(float(e) - float(t)), 3)}", file=out)
    return np.column_stack([est, true, np.abs(est - true)])
