"""Replica batches on the GPU (erirt_create_batch): replica r of a batch is the chain of a standalone engine with seed + r on
replica r's data and initial state -- every trace, the person and item / structural state and the running moments -- and the
evaluation, diagnostics, generated data (on an engine and through sampleBatch) and the batched runSimulation agree with their
standalone counterparts.  A write of one replica into another's copy of a buffer shows up in those comparisons; the guard zones
(ERIRT_GUARDS=1) follow each whole buffer and catch writes past the last replica."""
import numpy as np
import pytest

from helpers import make_problem

pytestmark = pytest.mark.gpu

FIVE = ["MlIrt", "RtIrt", "RtIrtNull", "RtIrtLatent", "RtIrtLatentQr"]
TOL = {"f64": 1e-10, "f32": 1e-5}  # as test_checkpoint_resume_is_bit_exact
SEED = 99


def _init(pb):
    init, model = pb["init"], pb["model"]
    st = dict(theta=init["theta"], a=init["a"], b=init["b"])
    if model != "MlIrt":
        st.update(zeta=init["zeta"], lambda_=init["lambda_"], sigma2=init["sigma2"], Sigma=init["Sigma"])
    if pb["nb"]:
        st["beta"] = init["beta"][: pb["nb"]]
    return st


def _engine(E, pb, dtype, n_iter, n_chain=1, n_burnin=2, seed=SEED, n_batch=1):
    model = pb["model"]
    return E.Engine(model, pb["N"], pb["J"], pb["F"], n_iter=n_iter, n_chain=n_chain, n_burnin=n_burnin, q_rt=pb["q"], dtype=dtype,
                    seed=seed, cov2one=model not in ("RtIrtLatent", "RtIrtLatentQr"), person_trace=False, use_graph=True,
                    n_batch=n_batch)


def _standalone(E, pb, dtype, sweeps, seed, **kw):
    eng = _engine(E, pb, dtype, sweeps // kw.get("n_chain", 1), seed=seed, **kw)
    eng.set_data(pb["Y"], None if pb["model"] == "MlIrt" else pb["logT"], pb["X"] if pb["F"] > 0 else None)
    eng.set_state(**_init(pb))
    eng.sample(sweeps)
    return eng


def _batch(E, pbs, dtype, sweeps, **kw):
    pb0 = pbs[0]
    eng = _engine(E, pb0, dtype, sweeps // kw.get("n_chain", 1), n_batch=len(pbs), **kw)
    eng.set_data(np.stack([p["Y"] for p in pbs]), None if pb0["model"] == "MlIrt" else np.stack([p["logT"] for p in pbs]),
                 np.stack([p["X"] for p in pbs]) if pb0["F"] > 0 else None)
    inits = [_init(p) for p in pbs]
    eng.set_state(**{k: [i[k] for i in inits] for k in inits[0]})
    eng.sample(sweeps)
    return eng


def _fields(pb):
    model = pb["model"]
    f = ["theta", "a", "b"] + (["zeta", "lambda", "sigma2", "Sigma"] if model != "MlIrt" else [])
    f += ["beta"] if pb["nb"] else []
    f += ["nu"] if model == "RtIrtLatentQr" else []
    return f


def _columns(eng, N):
    """(trace, first column, columns) of every traced column without a person trace: item columns of ra / rt, the structural
    columns of qr (LatentQr's trailing nu block is a person block), logLike"""
    out = [("ra", N, eng.trace_width("ra") - N), ("logLike", 0, 1)]
    if eng.model != 0:
        out.append(("rt", N, eng.trace_width("rt") - N))
    out.append(("qr", 0, eng.trace_width("qr") - (N if eng.model == 6 else 0)))
    return out


def _assert_replicas_equal_standalones(E, pbs, dtype, sweeps, **kw):
    tol = TOL[dtype]
    bat = _batch(E, pbs, dtype, sweeps, **kw)
    N = pbs[0]["N"]
    for r, pb in enumerate(pbs):
        one = _standalone(E, pb, dtype, sweeps, SEED + r, **kw)
        for which, c0, n in _columns(one, N):
            np.testing.assert_allclose(bat.get_trace(which, c0, n)[r], one.get_trace(which, c0, n), rtol=tol, atol=tol,
                                       err_msg=f"{which} replica {r}")
        for name in _fields(pb):
            np.testing.assert_allclose(bat.get_state(name)[r], np.asarray(one.get_state(name)).reshape(np.shape(bat.get_state(name)[r])),
                                       rtol=tol, atol=tol, err_msg=f"{name} replica {r}")
        for name in ["theta"] + (["zeta"] if pb["model"] != "MlIrt" else []) + (["nu"] if pb["model"] == "RtIrtLatentQr" else []):
            (bm, bs), (om, os_) = bat.get_moments(name), one.get_moments(name)
            np.testing.assert_allclose(bm[r], om, rtol=tol, atol=tol)
            np.testing.assert_allclose(bs[r], os_, rtol=tol, atol=tol)
        one.close()
    return bat


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("N", [100, 300])
@pytest.mark.parametrize("model", FIVE)
def test_replica_equals_standalone_handle(model, N, dtype):
    import erirt_b200 as E
    pbs = [make_problem(model, N, 7, 2, seed=10 + r) for r in range(3)]
    bat = _assert_replicas_equal_standalones(E, pbs, dtype, 6)
    ra = bat.get_trace("ra", N)
    assert not np.allclose(ra[0], ra[1]) and not np.allclose(ra[1], ra[2])  # the replicas are different chains
    bat.close()


def test_several_tiles_per_cta(monkeypatch):
    """A grid capped far below the tile count (ERIRT_MAX_GRID) gives every CTA of a replica many tiles: the dynamic tile dealing
    and the cross-tile accumulators run per replica."""
    import erirt_b200 as E
    monkeypatch.setenv("ERIRT_MAX_GRID", "4")
    pbs = [make_problem("RtIrt", 20000, 9, 2, seed=40 + r) for r in range(2)]
    _assert_replicas_equal_standalones(E, pbs, "f64", 4).close()


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_evaluation_diagnostics_and_trace_layout(dtype):
    import erirt_b200 as E
    pbs = [make_problem("RtIrtLatentQr", 200, 7, 2, seed=60 + r) for r in range(3)]
    sweeps, n_chain = 60, 3
    bat = _batch(E, pbs, dtype, sweeps, n_chain=n_chain, n_burnin=4)
    ll = bat.loglik_current()
    assert ll.shape == (3,)
    ess, rhat = bat.trace_ess_rhat("ra", 200, 14, skip=4)
    assert ess.shape == (3, 14)
    tr = bat.get_trace("ra", 200)
    assert tr.shape == (3, sweeps // n_chain, 14, n_chain)
    for r, pb in enumerate(pbs):
        one = _standalone(E, pb, dtype, sweeps, SEED + r, n_chain=n_chain, n_burnin=4)
        tol = TOL[dtype]
        assert abs(ll[r] - one.loglik_current()) <= tol * abs(ll[r])
        e1, r1 = one.trace_ess_rhat("ra", 200, 14, skip=4)
        np.testing.assert_allclose(ess[r], e1, rtol=1e-6)
        np.testing.assert_allclose(rhat[r], r1, rtol=1e-8)
        np.testing.assert_allclose(tr[r], one.get_trace("ra", 200), rtol=tol, atol=tol)
        one.close()
    bat.close()


@pytest.mark.parametrize("model", ["RtIrt", "MlIrt"])
def test_generated_data_equals_standalone_generator(model):
    import erirt_b200 as E
    B, N, J, F = 3, 257, 7, 2
    rng = np.random.default_rng(5)
    th, ze, X = rng.normal(size=(B, N)), rng.normal(size=(B, N)), rng.normal(size=(B, N, F))
    a, b, lam, s2 = rng.uniform(0.5, 1.5, (B, J)), rng.normal(size=(B, J)), 3 + rng.normal(size=(B, J)), rng.uniform(0.2, 1, (B, J))
    rt = model != "MlIrt"
    kw = dict(n_iter=2, q_rt=0.5, dtype="f64", person_trace=False)
    bat = E.Engine(model, N, J, F, n_batch=B, **kw)
    bat.generate_data(th, a, b, ze if rt else None, lam if rt else None, s2 if rt else None, None, X, error="tnorm", seed=77)
    Yb, Tb = bat.get_data()
    for r in range(B):
        one = E.Engine(model, N, J, F, **kw)
        one.generate_data(th[r], a[r], b[r], ze[r] if rt else None, lam[r] if rt else None, s2[r] if rt else None, None, X[r],
                          error="tnorm", seed=77 + r)
        Y1, T1 = one.get_data()
        assert np.array_equal(Yb[r], Y1)
        if rt:
            np.testing.assert_allclose(Tb[r], T1, rtol=1e-12, atol=1e-12)
        one.close()
    bat.close()


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_guard_zones_stay_clean(monkeypatch, dtype):
    """Nothing is written past the last replica's copy of any buffer (the zones do not sit between replicas)."""
    import erirt_b200 as E
    monkeypatch.setenv("ERIRT_GUARDS", "1")
    pbs = [make_problem("RtIrtLatentQr", 300, 9, 2, seed=80 + r) for r in range(4)]
    bat = _batch(E, pbs, dtype, 20)
    bat.loglik_current()
    assert bat.check_guards() == 0
    bat.close()


def test_run_simulation_batches_reproduce_the_sequential_dict():
    from erirt_b200 import api, simtools, simulate, structs
    C = structs.setCond(nSubj=150, nItem=6, nFeat=2, nIter=40, nChain=2, nRep=4)
    rng = np.random.default_rng(3)
    tp = structs.InputPara(a=rng.uniform(0.7, 1.4, 6), b=rng.normal(0, 0.5, 6), lambda_=3 + rng.normal(0, 0.3, 6),
                           sigma2t=rng.uniform(0.2, 0.5, 6), beta=rng.normal(0, 0.5, (2, 2)), Sigma_p=np.array([[1, 0.3], [0.3, 0.5]]))
    kw = dict(Para=("a", "b", "λ", "σ²t", "β"), funcData=simulate.setDataRtIrt, funcGibbs=api.GibbsRtIrt, seed=11, dtype="f64",
              person_trace=False)
    ref = simtools.runSimulation(C, tp, **kw)
    for batch in (4, 3):
        got = simtools.runSimulation(C, tp, batch=batch, **kw)
        assert sorted(got, key=str) == sorted(ref, key=str)
        for run in range(1, 5):
            for p in kw["Para"]:
                np.testing.assert_allclose(got[run][p], ref[run][p], rtol=1e-8, atol=1e-8)
            np.testing.assert_allclose(got[run]["Dic"], ref[run]["Dic"], rtol=1e-8)
            assert got[run]["Diag"]["essN"] == ref[run]["Diag"]["essN"] and got[run]["Diag"]["rhatN"] == ref[run]["Diag"]["rhatN"]


def _device_models(n, seed0):
    from erirt_b200 import api, simulate, structs
    C = structs.setCond(nSubj=300, nItem=8, nFeat=2, nIter=30, nChain=2)
    out = []
    for r in range(n):
        tp = simulate.setTrueParaRtIrt(C, rng=5)
        D = simulate.setDataOnDevice(C, tp, "RtIrt", rng=20 + r, seed=seed0 + r)
        out.append(api.GibbsRtIrt(C, Data=D, truePara=tp, rng=40 + r))
    return out


def test_sample_batch_on_device_data_equals_sample():
    """sampleBatch with DeviceData replicas (one stacked generate_data call, data seeds seed_0 + r) and getDicBatch give what
    sample and getDic give for each replica."""
    from erirt_b200 import api
    bat = api.sampleBatch(_device_models(2, 500), seed=11)
    dics = api.getDicBatch(bat)
    for r, M in enumerate(_device_models(2, 500)):
        api.sample(M, seed=11 + r, person_trace=False)
        B = bat[r]
        for name in ("ra", "rt", "qr", "logLike"):
            np.testing.assert_allclose(getattr(B.Post, name), getattr(M.Post, name), rtol=1e-10, atol=1e-10, err_msg=name)
        for f in ("theta", "zeta", "a", "b", "lambda_", "sigma2t", "beta", "Sigma_p"):
            np.testing.assert_allclose(getattr(B.Post.mean, f), getattr(M.Post.mean, f), rtol=1e-10, atol=1e-10, err_msg=f)
            np.testing.assert_allclose(getattr(B.Para, f), getattr(M.Para, f), rtol=1e-10, atol=1e-10, err_msg=f)
        np.testing.assert_allclose(dics[r].DIC, api.getDic(M).DIC, rtol=1e-10)
    assert not np.allclose(bat[0].Post.ra, bat[1].Post.ra)


def test_per_chain_entry_points_refuse_a_batch():
    import erirt_b200 as E
    pbs = [make_problem("RtIrt", 100, 5, 1, seed=90 + r) for r in range(2)]
    bat = _batch(E, pbs, "f64", 2)
    for call in (bat.checkpoint, lambda: bat.restore(np.zeros(64, np.uint8)), lambda: bat.comm_init(0, 2),
                 bat.peer_export, lambda: bat.peer_attach(b"\0" * 128), bat.peer_detach):
        with pytest.raises(E.ErirtError) as ei:
            call()
        assert ei.value.code == -5 and "replica batch" in str(ei.value)
    bat.close()
