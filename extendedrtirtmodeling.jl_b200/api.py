"""Host-side mirror of the reference's sampler API for the hot path (SURVEY.md 8b):

    Cond = setCond(nSubj=1000, nItem=15)
    MCMC = GibbsMlIrt(Cond, Data=Data, truePara=truePara)      # README.md:70
    sample(MCMC)                                               # sample!(MCMC), README.md:71
    MCMC.Post.mean.b                                           # README.md:74

Constructors draw the initial values exactly like setInitialValues (src/GibbsRtIrt.pl.jl:84-133,
src/GibbsRtIrtCross.pl.jl:85-134, src/GibbsRtIrtLatent.pl.jl:78-124) and `sample` replaces the body of the
sample! methods by calls into the C ABI (include/erirt_b200.h); the Julia package binds the same ABI through
ccall (julia/ErirtB200.jl).  There is no CPU path here.
"""
import numpy as np

from . import _lib
from .engine import Engine
from .simulate import DeviceData
from .structs import InputPara, OutputDic, OutputPost

# budget for keeping the full person-level trace on the device/host (bytes); beyond it Post.ra / Post.rt hold
# the item columns only and person parameters are summarised by running moments (SURVEY 0.10)
PERSON_TRACE_BUDGET = 2 << 30


class _GibbsBase:
    model = None            # key of _lib.MODELS
    default_cov2one = True  # sample! keyword default
    has_rt = True

    def __init__(self, Cond, Data=None, truePara=None, rng=None):
        self.Cond, self.Data, self.truePara = Cond, Data, truePara
        self.Para = None
        self.Post = OutputPost()
        self._rng = rng if isinstance(rng, np.random.Generator) else np.random.default_rng(rng)
        self.setInitialValues()
        self.engine = None

    def _base_init(self):
        C = self.Cond
        return dict(theta=self._rng.standard_normal(C.nSubj), a=np.ones(C.nItem), b=np.zeros(C.nItem))

    def _rt_init(self):
        C = self.Cond
        return dict(zeta=self._rng.standard_normal(C.nSubj), lambda_=np.zeros(C.nItem), sigma2t=np.ones(C.nItem),
                    Sigma_p=np.eye(2))


class GibbsMlIrt(_GibbsBase):
    """src/GibbsRtIrt.pl.jl:76-106"""
    model, has_rt = "MlIrt", False

    def setInitialValues(self):
        self.Para = InputPara(**self._base_init(), beta=self._rng.standard_normal(self.Cond.nFeat + 1))


class GibbsRtIrt(_GibbsBase):
    """src/GibbsRtIrt.pl.jl:114-146"""
    model = "RtIrt"

    def setInitialValues(self):
        self.Para = InputPara(**self._base_init(), **self._rt_init(),
                              beta=self._rng.standard_normal((self.Cond.nFeat + 1, 2)))


class GibbsRtIrtNull(_GibbsBase):
    """src/GibbsRtIrt.pl.jl:151-183"""
    model = "RtIrtNull"

    def setInitialValues(self):
        self.Para = InputPara(**self._base_init(), **self._rt_init())


class GibbsRtIrtCross(_GibbsBase):
    """src/GibbsRtIrtCross.pl.jl:77-110"""
    model = "RtIrtCross"

    def setInitialValues(self):
        self.Para = InputPara(**self._base_init(), **self._rt_init(), rho=self._rng.standard_normal(self.Cond.nItem))


class GibbsRtIrtCrossQr(GibbsRtIrtCross):
    """src/GibbsRtIrtCross.pl.jl:115-147"""
    model = "RtIrtCrossQr"


class GibbsRtIrtLatent(_GibbsBase):
    """src/GibbsRtIrtLatent.pl.jl:70-102"""
    model, default_cov2one = "RtIrtLatent", False

    def setInitialValues(self):
        self.Para = InputPara(**self._base_init(), **self._rt_init(), beta=self._rng.standard_normal(self.Cond.nFeat + 2))


class GibbsRtIrtLatentQr(GibbsRtIrtLatent):
    """src/GibbsRtIrtLatent.pl.jl:105-137"""
    model = "RtIrtLatentQr"


class GibbsRtIrtQuantile(GibbsRtIrtLatentQr):
    """README.md:95 names GibbsRtIrtQuantile; the snapshot only ships the LatentQr sampler behind that role
    (src/ExtendedRtIrtModeling.jl:65 has the export commented out).  Alias, see SURVEY.md 0.2."""


def _qr_layout(MCMC):
    C = MCMC.Cond
    p = C.nFeat + 1
    return {"MlIrt": [("beta", p)], "RtIrt": [("beta", 2 * p), ("Sigma_p", 4)], "RtIrtNull": [("beta", 2 * p), ("Sigma_p", 4)],
            "RtIrtCross": [("rho", C.nItem), ("Sigma_p", 4)], "RtIrtCrossQr": [("rho", C.nItem), ("Sigma_p", 4)],
            "RtIrtLatent": [("beta", C.nFeat + 2), ("Sigma_p", 4)], "RtIrtLatentQr": [("beta", C.nFeat + 2), ("Sigma_p", 4)]}[MCMC.model]


def sample(MCMC, intercept=False, itemtype="2pl", cov2one=None, *, dtype="f64", seed=1234, chain=0, device=0,
           person_trace=None, compat=0, use_graph=True, shard=None, progress=None, chunk=None, nu_cell_moments=None):
    """sample!(MCMC; intercept, itemtype, cov2one) for every Gibbs* type.

    Extra keyword-only engine options: dtype ("f64" parity mode / "f32" fast mode), seed, chain (independent
    chain id), device, person_trace, compat (quirk switches, default = as written in the reference),
    shard = (rank, world, nccl_unique_id_bytes, subj_offset, n_subj_total[, allgather]) for a person-sharded chain; the
    optional sixth entry is a callable bytes -> concatenated bytes of all ranks (e.g. distributed.allgather_bytes), which
    switches the per-sweep exchange from ncclAllReduce to the fused peer-memory all-reduce.
    nu_cell_moments (CrossQr): keep the running mean / SD of the N x J weights on the device so that Post.mean.ν exists
    (src/GibbsRtIrtCross.pl.jl:310) without the reference's nIter x N*J trace; default: on while 16 N J bytes fit the budget.
    Returns MCMC (mutated), like the reference."""
    if itemtype not in ("1pl", "2pl"):
        raise ValueError("Invalid input: the item type must be '1pl' or '2pl'.")  # src/GibbsRtIrt.pl.jl:212-214
    C, D, P0 = MCMC.Cond, MCMC.Data, MCMC.Para
    if cov2one is None:
        cov2one = MCMC.default_cov2one
    N, J, F = C.nSubj, C.nItem, C.nFeat
    n_sweeps = C.nIter * C.nChain
    if person_trace is None:
        person_trace = n_sweeps * N * 8 * 3 <= PERSON_TRACE_BUDGET
    n_total, offset = N, 0
    if shard is not None:
        offset, n_total = shard[3], shard[4]
    if nu_cell_moments is None:
        nu_cell_moments = MCMC.model == "RtIrtCrossQr" and 16 * N * J <= PERSON_TRACE_BUDGET
    eng = Engine(MCMC.model, N, J, F, n_iter=C.nIter, n_chain=C.nChain, n_burnin=C.nBurnin, q_rt=C.qRt,
                 intercept=intercept, itemtype=itemtype, cov2one=cov2one, dtype=dtype, seed=seed, chain=chain,
                 compat=compat, person_trace=person_trace, device=device, use_graph=use_graph,
                 n_subj_total=n_total, subj_offset=offset, nu_cell_moments=nu_cell_moments and MCMC.model == "RtIrtCrossQr")
    MCMC.nu_cell_moments = bool(nu_cell_moments and MCMC.model == "RtIrtCrossQr")
    MCMC.engine = eng
    if shard is not None:
        eng.comm_init(shard[0], shard[1], shard[2])
        if len(shard) > 5 and shard[5] is not None:
            eng.peer_attach(shard[5](eng.peer_export()))
    if isinstance(D, DeviceData):  # the N x J part is generated on the device (a shard generates its rows of the one data set)
        D.generate_into(eng, MCMC.has_rt, offset, offset + N) if shard is not None and len(D.truePara.theta) == n_total \
            else D.generate_into(eng, MCMC.has_rt)
    else:
        eng.set_data(D.Y, D.logT if MCMC.has_rt else None, D.X if F > 0 else None)
    init = dict(theta=P0.theta, a=P0.a, b=P0.b)
    if MCMC.has_rt:
        init.update(zeta=P0.zeta, lambda_=P0.lambda_, sigma2=P0.sigma2t, Sigma=P0.Sigma_p)
    if P0.beta.size:
        init["beta"] = P0.beta
    if P0.rho.size:
        init["rho"] = P0.rho
    eng.set_state(**init)
    if chunk is None or progress is None:
        eng.sample(n_sweeps)
    else:  # the reference wraps the loop in @showprogress; the shim can drive a progress bar by chunks
        done = 0
        while done < n_sweeps:
            step = min(chunk, n_sweeps - done)
            eng.sample(step)
            done += step
            progress(done, n_sweeps)
    _collect(MCMC, eng, person_trace)
    return MCMC


def _collect(MCMC, eng, person_trace):
    C = MCMC.Cond
    N, J = C.nSubj, C.nItem
    Post = MCMC.Post
    Post.person_cols = bool(person_trace)
    c0 = 0 if person_trace else N
    Post.ra = eng.get_trace("ra", c0, N + 2 * J - c0)
    Post.rt = eng.get_trace("rt", c0, N + 2 * J - c0) if MCMC.has_rt else None
    qw_small = sum(n for _, n in _qr_layout(MCMC))
    qw = eng.trace_width("qr")
    Post.qr = eng.get_trace("qr", 0, qw if person_trace else qw_small)
    Post.logLike = eng.get_trace("logLike")
    nb = C.nBurnin
    mean = InputPara()
    sd = InputPara()

    def pm(arr, lo, hi):  # mean over [(nBurnin+1):end, lo:hi, all chains]   src/GibbsRtIrt.pl.jl:327-343
        return arr[nb:, lo:hi, :].mean(axis=(0, 2))

    o = 0
    for name, n in _qr_layout(MCMC):
        setattr(mean, name, pm(Post.qr, o, o + n))
        o += n
    ic = N - c0  # first item column inside the returned ra/rt
    mean.a, mean.b = pm(Post.ra, ic, ic + J), pm(Post.ra, ic + J, ic + 2 * J)
    if MCMC.has_rt:
        mean.lambda_, mean.sigma2t = pm(Post.rt, ic, ic + J), pm(Post.rt, ic + J, ic + 2 * J)
    if person_trace:
        mean.theta = pm(Post.ra, 0, N)
        if MCMC.has_rt:
            mean.zeta = pm(Post.rt, 0, N)
        if MCMC.model == "RtIrtLatentQr":
            mean.nu = pm(Post.qr, qw_small, qw_small + N)
    m, s = eng.get_moments("theta")
    sd.theta = s
    if not person_trace:
        mean.theta = m
    if MCMC.has_rt:
        m, s = eng.get_moments("zeta")
        sd.zeta = s
        if not person_trace:
            mean.zeta = m
    if MCMC.model == "RtIrtLatentQr":
        m, s = eng.get_moments("nu")
        sd.nu = s
        if not person_trace:
            mean.nu = m
    if MCMC.model == "RtIrtCrossQr" and getattr(MCMC, "nu_cell_moments", False):
        mean.nu, sd.nu = eng.get_moments("nu")  # N x J, src/GibbsRtIrtCross.pl.jl:310
    Post.mean, Post.sd = mean, sd
    # The reference leaves the COMPLETE last state in MCMC.Para, so a second sample!(MCMC) continues the chain.  The engine pipelines
    # the person draws of sweep n with the item / structural draws of sweep n+1 (erirt_b200.h, erirt_set_state), so the item and
    # structural fields of state n are the LAST TRACE ROW, not erirt_get_state.
    Para = MCMC.Para
    Para.theta = eng.get_state("theta")
    if MCMC.has_rt:
        Para.zeta = eng.get_state("zeta")
    last = (C.nIter - 1, slice(None), C.nChain - 1)
    ra_last, qr_last = Post.ra[last], Post.qr[last]
    Para.a, Para.b = ra_last[ic:ic + J].copy(), ra_last[ic + J:ic + 2 * J].copy()
    if MCMC.has_rt:
        rt_last = Post.rt[last]
        Para.lambda_, Para.sigma2t = rt_last[ic:ic + J].copy(), rt_last[ic + J:ic + 2 * J].copy()
    o = 0
    for name, n in _qr_layout(MCMC):
        v = qr_last[o:o + n].copy()
        cur = getattr(Para, name, None)
        if cur is not None and np.size(cur) == n and np.ndim(cur) > 1:
            v = v.reshape(np.shape(cur), order="F")  # beta keeps its (nFeat+1) x 2 shape, Sigma_p its 2 x 2
        setattr(Para, name, v)
        o += n


sample_bang = sample  # `sample!` is not a Python identifier


class _ReplicaView:
    """Replica r of a batched engine seen through the getters _collect uses; each batched read is made once and shared by the views."""

    def __init__(self, eng, r, cache):
        self.eng, self.r, self.cache = eng, r, cache

    def _get(self, *key):
        if key not in self.cache:
            self.cache[key] = getattr(self.eng, key[0])(*key[1:])
        return self.cache[key]

    def _at(self, v):
        return v[self.r] if self.eng.B > 1 else v  # a batch of one has the standalone shapes

    def trace_width(self, which):
        return self.eng.trace_width(which)

    def get_trace(self, which, first_col=0, n_cols=None):
        return self._at(self._get("get_trace", which, first_col, n_cols))

    def get_moments(self, name):
        m, s = self._get("get_moments", name)
        return self._at(m), self._at(s)

    def get_state(self, name):
        return self._at(self._get("get_state", name))


def _check_batch(MCMCs, person_trace=False):
    """ValueError (before any GPU work) unless MCMCs can share one replica batch."""
    if len(MCMCs) == 0:
        raise ValueError("sampleBatch needs at least one model object")
    M0 = MCMCs[0]
    if any(type(M) is not type(M0) for M in MCMCs):
        raise ValueError("sampleBatch: all model objects must be of one type")
    if any(M.Cond != M0.Cond for M in MCMCs):
        raise ValueError("sampleBatch: all model objects must have equal Cond")
    if M0.model in ("RtIrtCross", "RtIrtCrossQr"):
        raise ValueError("sampleBatch: the Cross family is not supported (two-stage sweep)")
    if person_trace:
        raise ValueError("sampleBatch keeps no person trace (person_trace=True is not supported)")
    dev = [isinstance(M.Data, DeviceData) for M in MCMCs]
    if any(dev) and not all(dev):
        raise ValueError("sampleBatch: mixed host and device data")
    if all(dev):
        D0 = M0.Data
        if any(M.Data.error != D0.error or M.Data.seed != D0.seed + r or (M.Data.X is None) != (D0.X is None) for r, M in enumerate(MCMCs)):
            raise ValueError("sampleBatch: device data of a batch must share the error type, and replica r must have data seed seed_0 + r")


def _batch_data(eng, MCMCs):
    M0, F = MCMCs[0], MCMCs[0].Cond.nFeat
    if isinstance(M0.Data, DeviceData):  # one call: replica r generates with data seed D_0.seed + r
        P = [M.Data.truePara for M in MCMCs]
        cat = lambda f: np.concatenate([np.asarray(f(p), dtype=np.float64).ravel() for p in P])  # noqa: E731
        has_rt = M0.has_rt
        eng.generate_data(cat(lambda p: p.theta), cat(lambda p: p.a), cat(lambda p: p.b), cat(lambda p: p.zeta) if has_rt else None,
                          cat(lambda p: p.lambda_) if has_rt else None,
                          cat(lambda p: p.sigma2t) if (has_rt and np.size(P[0].sigma2t)) else None,
                          cat(lambda p: p.rho) if np.size(P[0].rho) else None,
                          None if M0.Data.X is None else np.concatenate([M.Data.X for M in MCMCs], axis=0),
                          error=M0.Data.error, seed=M0.Data.seed)
    else:
        eng.set_data(np.concatenate([np.asarray(M.Data.Y) for M in MCMCs], axis=0),
                     np.concatenate([M.Data.logT for M in MCMCs], axis=0) if M0.has_rt else None,
                     np.concatenate([M.Data.X for M in MCMCs], axis=0) if F > 0 else None)


def sampleBatch(MCMCs, intercept=False, itemtype="2pl", cov2one=None, *, seed=1234, dtype="f64", chain=0, device=0,
                person_trace=False, compat=0, use_graph=True):
    """sample(MCMC_r, seed=seed + r, person_trace=False) for every MCMC_r of `MCMCs`, as ONE replica batch on one GPU
    (erirt_create_batch, DESIGN.md 6.6): one person launch and one global launch per sweep for all of them.  The model objects
    must be of one type (not the Cross family) with equal Cond; each brings its own Data (all host InputData, or all DeviceData with
    consecutive data seeds) and initial Para.  Fills every MCMC.Post and MCMC.Para exactly as the sequential calls would.
    Returns MCMCs."""
    if itemtype not in ("1pl", "2pl"):
        raise ValueError("Invalid input: the item type must be '1pl' or '2pl'.")
    MCMCs = list(MCMCs)
    _check_batch(MCMCs, person_trace)
    M0 = MCMCs[0]
    C = M0.Cond
    if cov2one is None:
        cov2one = M0.default_cov2one
    eng = Engine(M0.model, C.nSubj, C.nItem, C.nFeat, n_iter=C.nIter, n_chain=C.nChain, n_burnin=C.nBurnin, q_rt=C.qRt,
                 intercept=intercept, itemtype=itemtype, cov2one=cov2one, dtype=dtype, seed=seed, chain=chain, compat=compat,
                 person_trace=False, device=device, use_graph=use_graph, n_batch=len(MCMCs))
    try:
        _batch_data(eng, MCMCs)
        P = [M.Para for M in MCMCs]
        init = dict(theta=[p.theta for p in P], a=[p.a for p in P], b=[p.b for p in P])
        if M0.has_rt:
            init.update(zeta=[p.zeta for p in P], lambda_=[p.lambda_ for p in P], sigma2=[p.sigma2t for p in P], Sigma=[p.Sigma_p for p in P])
        if P[0].beta.size:
            init["beta"] = [p.beta for p in P]
        eng.set_state(**init)
        eng.sample(C.nIter * C.nChain)
        cache = {}
        for r, M in enumerate(MCMCs):
            M.nu_cell_moments = False
            _collect(M, _ReplicaView(eng, r, cache), False)
    finally:
        eng.close()
    return MCMCs


def sampleIndependentChains(MCMC, n_chains, group=None, rng=0, **kw):
    """BASELINE configs[3] / SURVEY 8e "independent chains": n_chains truly independent chains of MCMC's model on MCMC's data -- distinct
    Philox keys (chain id c) and distinct initial values (constructor seeded rng + c) -- dealt to the ranks of the torch.distributed
    group c -> rank c mod world (one GPU each; a single process runs them one after the other), no collective while sampling.  The
    reference has only interleaved pseudo-chains (one state, `for m in 1:nIter, l in 1:nChain`, src/GibbsRtIrt.pl.jl:289), so this is
    new behaviour behind the same Post layout: MCMC.Post.ra / rt / qr / logLike come back as [nIter, item and structural columns,
    n_chains] (person columns are not gathered), Post.mean is the mean over chains of the per-chain means, and MCMC.Cond.nChain is
    set to n_chains, so precis / checkConvergence / getDic read it like any other run.  kw: sample()'s keyword arguments."""
    import dataclasses

    from .distributed import run_independent_chains
    C1 = dataclasses.replace(MCMC.Cond, nChain=1)
    for k in ("chain", "person_trace", "shard"):
        kw.pop(k, None)

    def run_chain(c):
        M = type(MCMC)(C1, Data=MCMC.Data, truePara=MCMC.truePara, rng=rng + c)
        sample(M, chain=c, person_trace=False, **kw)
        P = M.Post
        out = dict(ra=P.ra, qr=P.qr[:, :sum(n for _, n in _qr_layout(M)), :], logLike=P.logLike)
        if M.has_rt:
            out["rt"] = P.rt
        for f in InputPara._FIELDS:  # per-chain posterior means, chain axis last
            v = np.asarray(getattr(P.mean, f), dtype=np.float64)
            if v.size:
                out["mean_" + f] = v.reshape(v.shape + (1,))
        M.engine.close()
        return out

    res = run_independent_chains(run_chain, n_chains, group)
    MCMC.Cond = dataclasses.replace(MCMC.Cond, nChain=n_chains)
    Post = OutputPost()
    Post.ra, Post.qr, Post.logLike, Post.rt = res["ra"], res["qr"], res["logLike"], res.get("rt")
    Post.person_cols = False
    Post.mean = InputPara(**{k[5:]: v.mean(axis=-1) for k, v in res.items() if k.startswith("mean_")})
    MCMC.Post = Post
    return MCMC


def getLogLikelihood(MCMC, P, dtype="f64", device=0):
    """getLogLikelihood*(Cond, Data; P) (src/GibbsRtIrt.pl.jl:195-204, 262-272, 351-361; Cross :158-169; Latent :151-161,
    :243-264), evaluated on the GPU for an InputPara `P` (e.g. MCMC.Post.mean)."""
    C, D = MCMC.Cond, MCMC.Data
    eng = Engine(MCMC.model, C.nSubj, C.nItem, C.nFeat, n_iter=1, n_chain=1, q_rt=C.qRt, dtype=dtype, device=device,
                 person_trace=False, use_graph=False)
    try:
        if isinstance(D, DeviceData):
            D.generate_into(eng, MCMC.has_rt)
        else:
            eng.set_data(D.Y, D.logT if MCMC.has_rt else None, D.X if C.nFeat > 0 else None)
        st = dict(theta=P.theta, a=P.a, b=P.b)
        if MCMC.has_rt:
            st.update(zeta=P.zeta, lambda_=P.lambda_, sigma2=P.sigma2t, Sigma=np.asarray(P.Sigma_p).reshape(4))
        if P.beta.size:
            st["beta"] = P.beta
        if P.rho.size:
            st["rho"] = P.rho
        if MCMC.model in ("RtIrtLatentQr", "RtIrtCrossQr"):
            if np.size(P.nu) == 0:
                raise ValueError("the log-likelihood of a quantile model needs the weights ν (sample CrossQr with nu_cell_moments=True)")
            st["nu"] = P.nu
        eng.set_state(**st)
        return eng.loglik_current()
    finally:
        eng.close()


def getDic(MCMC, dtype="f64", device=0):
    """getDic (src/GibbsRtIrt.pl.jl:432-472): D-hat = -2 loglik(Post.mean), D-bar = -2 mean(Post.logLike) over ALL
    iterations including burn-in (quirk Q10), pD = D-bar - D-hat, DIC = D-bar + pD."""
    Dhat = -2.0 * getLogLikelihood(MCMC, MCMC.Post.mean, dtype=dtype, device=device)
    Dbar = -2.0 * float(np.mean(MCMC.Post.logLike))
    dic = OutputDic()
    dic.pD = Dbar - Dhat
    dic.DIC = Dbar + dic.pD
    return dic


def getDicBatch(MCMCs, dtype="f64", device=0):
    """getDic(MCMC_r) for every MCMC_r of `MCMCs` (one type, equal Cond, sampled), with ONE batched evaluation engine: one
    loglik_current call evaluates every replica's Post.mean on its own data."""
    MCMCs = list(MCMCs)
    _check_batch(MCMCs)
    M0 = MCMCs[0]
    C = M0.Cond
    eng = Engine(M0.model, C.nSubj, C.nItem, C.nFeat, n_iter=1, n_chain=1, q_rt=C.qRt, dtype=dtype, device=device,
                 person_trace=False, use_graph=False, n_batch=len(MCMCs))
    try:
        _batch_data(eng, MCMCs)
        P = [M.Post.mean for M in MCMCs]
        st = dict(theta=[p.theta for p in P], a=[p.a for p in P], b=[p.b for p in P])
        if M0.has_rt:
            st.update(zeta=[p.zeta for p in P], lambda_=[p.lambda_ for p in P], sigma2=[p.sigma2t for p in P],
                      Sigma=[np.asarray(p.Sigma_p).reshape(4) for p in P])
        if P[0].beta.size:
            st["beta"] = [p.beta for p in P]
        if M0.model == "RtIrtLatentQr":
            st["nu"] = [p.nu for p in P]
        eng.set_state(**st)
        ll = np.atleast_1d(eng.loglik_current())
    finally:
        eng.close()
    out = []
    for M, l in zip(MCMCs, ll):
        Dhat, Dbar = -2.0 * float(l), -2.0 * float(np.mean(M.Post.logLike))
        dic = OutputDic()
        dic.pD = Dbar - Dhat
        dic.DIC = Dbar + dic.pD
        out.append(dic)
    return out


def _param_names(MCMC):
    C = MCMC.Cond
    J, F = C.nItem, C.nFeat
    ra = [f"a{i}" for i in range(1, J + 1)] + [f"b{i}" for i in range(1, J + 1)]
    rt = [f"λ{i}" for i in range(1, J + 1)] + [f"σ²t{i}" for i in range(1, J + 1)]
    sig = ["Σ[1,1]", "Σ[1,2]", "Σ[2,1]", "Σ[2,2]"]
    qr = {"MlIrt": [f"β[{i}]" for i in range(F + 1)],
          "RtIrt": [f"β[{i},{j}]" for j in (1, 2) for i in range(F + 1)] + sig,
          "RtIrtNull": [f"β[{i},{j}]" for j in (1, 2) for i in range(F + 1)] + sig,
          "RtIrtCross": [f"ρ{i}" for i in range(1, J + 1)] + sig, "RtIrtCrossQr": [f"ρ{i}" for i in range(1, J + 1)] + sig,
          "RtIrtLatent": [f"β{i}" for i in range(F + 2)] + sig, "RtIrtLatentQr": [f"β{i}" for i in range(F + 2)] + sig}[MCMC.model]
    return ra, rt, qr


def precis(MCMC, file=None):
    """precis(MCMC) (src/GibbsRtIrt.pl.jl:607-675, src/Base.pl.jl:152-167): mean, std, ess, rhat, 2.5 % / 97.5 % quantiles of the
    item and structural parameters over the post-burn-in draws.  Returns the rows (list of dicts) and prints the tables."""
    from .diagnostics import summarize
    C, Post = MCMC.Cond, MCMC.Post
    nb, N = C.nBurnin, C.nSubj
    ic = N if Post.person_cols else 0
    ra_n, rt_n, qr_n = _param_names(MCMC)
    blocks = [("1) Item Response Model.", Post.ra[nb:, ic:ic + 2 * C.nItem, :], ra_n)]
    if MCMC.has_rt:
        blocks.append(("2) Response Time Model.", Post.rt[nb:, ic:ic + 2 * C.nItem, :], rt_n))
    blocks.append(("3) Structural Model.", Post.qr[nb:, :len(qr_n), :], qr_n))
    out = []
    for title, arr, names in blocks:
        rows = summarize(arr, names)
        out.extend(rows)
        print(title, file=file)
        print(f"{'':>10s} {'mean':>9s} {'std':>9s} {'ess':>9s} {'rhat':>7s} {'q025':>9s} {'q975':>9s}", file=file)
        for r in rows:
            sig = "" if (r["q025"] < 0 < r["q975"]) else "*"
            print(f"{r['name']:>10s} {r['mean']:9.3f} {r['std']:9.3f} {r['ess']:9.1f} {r['rhat']:7.3f} {r['q025']:9.3f} {r['q975']:9.3f} {sig}", file=file)
    return out


def coef(MCMC, file=None):
    """coef(MCMC) (src/GibbsRtIrt.pl.jl:479-601): posterior means of the item parameters, covariance, regression coefficients, DIC."""
    m = MCMC.Post.mean
    print(f">> Model: {type(MCMC).__name__}. {MCMC.Cond.nSubj} subjects, {MCMC.Cond.nItem} items, {MCMC.Cond.nFeat} features; "
          f"{MCMC.Cond.nChain} chains of {MCMC.Cond.nIter} iterations, first {MCMC.Cond.nBurnin} discarded.", file=file)
    print("1) Item Parameters.", file=file)
    for j in range(MCMC.Cond.nItem):
        row = f"{j + 1:5d} {m.a[j]:7.3f} {m.b[j]:7.3f}"
        if MCMC.has_rt:
            row += f" {m.lambda_[j]:7.3f} {m.sigma2t[j]:7.3f}"
        print(row, file=file)
    if MCMC.has_rt:
        print("2) Covariance of Person Parameters.", np.asarray(m.Sigma_p).reshape(2, 2).round(3).tolist(), file=file)
    if m.beta.size:
        print("3) Regression Coefficients.", np.round(m.beta, 3).tolist(), file=file)
    dic = getDic(MCMC) if (MCMC.model != "RtIrtCrossQr" or np.size(MCMC.Post.mean.nu)) else None
    if dic is not None:
        print(f"4) Criterion. Deviance {dic.DIC - dic.pD:.3f}  DIC {dic.DIC:.3f}", file=file)
    return dic
