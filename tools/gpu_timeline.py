"""Sweep timeline of the diagnostic build diag_timeline.so (ERIRT_TIMELINE_BUILD=1 python tools/make_tick_build.py): %globaltimer
stamps of the person launch P(k) and the global kernel G(k+1) per sweep.  usage: python tools/gpu_timeline.py [C5|C5s8|C1|C2|C3]"""
import ctypes, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
TICKS = bool(os.environ.get("TICKS"))  # TICKS=1: the clock64() phase timers of diag_tick.so instead of the timeline
os.environ["ERIRT_B200_LIB"] = os.path.join(ROOT, "diag_tick.so" if TICKS else "diag_timeline.so")
import numpy as np, torch
import erirt_b200 as E
import bench

which = sys.argv[1] if len(sys.argv) > 1 else "C5"
dev = torch.device("cuda", 0)
K = 48
if which.startswith("C5"):
    tp = bench.true_params()
    world = 8 if which == "C5s8" else 1  # C5s8: the shard of one of eight GPUs (no exchange: timing of the local part only)
    dY, dT, dX, off, n = bench.gen_shard_torch(tp, 0, world, dev)
    th, ze, be = bench.init_state(off, n)
    eng = E.Engine("RtIrtQuantile", n, bench.N_ITEM, bench.N_FEAT, n_iter=200, n_chain=1, n_burnin=0, q_rt=bench.Q_RT, cov2one=False,
                   dtype="f32", seed=1, person_trace=False, use_graph=True)
    eng.set_data_device(dY.data_ptr(), n, dT.data_ptr(), n, dX.data_ptr(), n)
    eng.set_state(theta=th, zeta=ze, beta=be)
else:
    rng = np.random.default_rng(3)
    if which == "C1":
        Cond = E.setCond(nSubj=1000, nItem=15, nFeat=3, nIter=200, nChain=1)
        D = E.setDataMlIrt(Cond, E.setTrueParaMlIrt(Cond, rng=1), rng=1)
        model, N, J, F, init = "MlIrt", 1000, 15, 3, dict(theta=rng.standard_normal(1000), beta=rng.standard_normal(4))
    elif which == "C2":
        Cond = E.setCond(nSubj=10_000, nItem=30, nFeat=3, nIter=200, nChain=1)
        D = E.setDataRtIrt(Cond, E.setTrueParaRtIrt(Cond, rng=1), rng=1)
        model, N, J, F = "RtIrt", 10_000, 30, 3
        init = dict(theta=rng.standard_normal(N), zeta=rng.standard_normal(N), beta=rng.standard_normal(8))
    elif which == "C4":
        Cond = E.setCond(nSubj=100_000, nItem=40, nFeat=0, nIter=200, nChain=1)
        D = E.setDataRtIrtNull(Cond, E.setTrueParaRtIrt(Cond, rng=1), rng=1)
        model, N, J, F = "RtIrtNull", 100_000, 40, 0
        init = dict(theta=rng.standard_normal(N), zeta=rng.standard_normal(N))
    else:
        Cond = E.setCond(nSubj=631, nItem=14, nFeat=10, nIter=200, nChain=1, qRt=0.85)
        D = E.setDataRtIrtLatent(Cond, E.setTrueParaRtIrtLatent(Cond, rng=1), type="norm", rng=1)
        model, N, J, F = "RtIrtLatentQr", 631, 14, 10
        init = dict(theta=rng.standard_normal(N), zeta=rng.standard_normal(N), beta=rng.standard_normal(12))
    eng = E.Engine(model, N, J, F, n_iter=200, n_chain=1, n_burnin=0, q_rt=0.85, cov2one=(model != "RtIrtLatentQr"), dtype="f32", seed=1,
                   person_trace=False, use_graph=True)
    eng.set_data(D.Y, None if model == "MlIrt" else D.logT, D.X if F > 0 else None)
    eng.set_state(**init)
eng.sample(40)
if TICKS:
    tb = (ctypes.c_ulonglong * 16)()
    eng.lib.erirt_diag_ticks(tb, 1)
    eng.sample(K)
    eng.lib.erirt_diag_ticks(tb, 0)
    t = np.array(list(tb), dtype=np.float64)
    st = eng.stats()
    print(which, "ms per sweep", st["last_sample_ms"] / K, "deferred PG fraction", st.get("pg_deferred_frac"), "tpp", st.get("tpp"), "grid", st.get("grid"))
    names = ["issue+person part1", "mbar wait (TMA)", "row sums", "-", "person part 2 + u rows", "-", "PG main pass", "queue push", "barrier 3", "drain",
             "barrier 4", "statistics pass", "flush + Gram", "loop top / store issue", "-", "-"]
    tot = t.sum()
    for nm, v in zip(names, t):
        if v: print(f"  {nm:28s} {v / K:14.0f} warp-cycles per sweep  {100 * v / tot:5.1f} %")
    sys.exit(0)
eng.sample(K)
print(which, "ms per sweep", eng.stats()["last_sample_ms"] / K)
buf = (ctypes.c_ulonglong * (256 * 16))()
eng.lib.erirt_diag_timeline(buf)
t = np.array(list(buf), dtype=np.float64).reshape(256, 16)
ks = np.arange(48, 40 + K - 2)  # sweeps well inside the second sample() call
names = ["P first CTA entry", "P first CTA past wait", "P last CTA past wait", "P last CTA done", "G entry", "G pre-wait part done",
         "G past wait", "G statistics staged", "G log-likelihood done", "G draws done", "G end"]
rows = []
for k in ks:
    base = t[k, 0]
    rows.append([(t[k, i] - base) / 1e3 for i in range(11)] + [(t[k + 1, 0] - base) / 1e3, (t[k + 1, 2] - base) / 1e3] +
                [(t[k, i] - base) / 1e3 for i in (13, 11, 12, 14)])
m = np.median(np.array(rows), axis=0)
for nm, v in zip(names + ["next P first CTA entry", "next P last CTA past wait", "G  prebuild done", "G  structural warp done", "G  item lane 32 done",
                          "G  item lane 255 done"], m):
    print(f"  {nm:28s} {v:9.2f} us")

if os.environ.get("TL_CTAS"):
    cb = (ctypes.c_ulonglong * (1024 * 6))()
    eng.lib.erirt_diag_cta_timeline(cb)
    c = np.array(list(cb), dtype=np.float64).reshape(1024, 6)
    c = c[c[:, 1] > 0]
    t0 = c[:, 1].min()
    print("per-CTA view of sweep 60:", len(c), "CTAs on", len(set(c[:, 0])), "SMs")
    print("  past wait: min %.2f max %.2f us" % (0.0, (c[:, 1].max() - t0) / 1e3))
    end = (c[:, 3] - t0) / 1e3
    print("  end: quantiles", np.round(np.quantile(end, [0, .1, .5, .8, .9, .99, 1]), 1))
    pro = (c[:, 2] - c[:, 1]) / 1e3
    loop = (c[:, 4] - c[:, 2]) / 1e3
    epi = (c[:, 3] - c[:, 4]) / 1e3
    print("  prologue (wait -> tile loop): median %.2f max %.2f us; tile loop: median %.2f max %.2f us (tiles per CTA: median %d, max %d); epilogue (loop end -> CTA end): median %.2f max %.2f us"
          % (np.median(pro), pro.max(), np.median(loop), loop.max(), np.median(c[:, 5]), c[:, 5].max(), np.median(epi), epi.max()))
    late = end > np.quantile(end, 0.8)
    sm_counts = {}
    for smid in c[late, 0]: sm_counts[int(smid)] = sm_counts.get(int(smid), 0) + 1
    hist = {}
    for v in sm_counts.values(): hist[v] = hist.get(v, 0) + 1
    print("  CTAs in the slowest 20 %% per SM (count of SMs by how many such CTAs they hold):", hist)
    print("  block 0..7 -> SM", [int(x) for x in c[:8, 0]], " blocks 148..151 -> SM", [int(x) for x in c[148:152, 0]])
