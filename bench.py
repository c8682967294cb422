#!/usr/bin/env python
"""Benchmark of the Gibbs sweep path (BASELINE.json metric: "Gibbs sweeps/sec & ESS/sec, nSubj=1M nItem=100").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one Gibbs sweep of GibbsRtIrtQuantile (the LatentQr sampler, q = 0.85, F = 3 covariates) over the
synthetic BASELINE config 5: nSubj = 1,000,000 x nItem = 100, data from setDataRtIrtLatent(type="skew")
(src/SimTools.jl:300-343), f32 storage / per-cell arithmetic, f64 statistics, log-likelihood and running
person moments ON (the reference computes logLike and stores the trace every sweep).  With N > 1 the persons of
the one chain are sharded over the N GPUs of the box and the item statistics are all-reduced every sweep (one-shot
exchange over NVLink peer memory fused into the global draw kernel; ERIRT_EXCHANGE=nccl selects ncclAllReduce), so
the total work is fixed: "scaling": "strong".

Keys of the JSON line (DESIGN.md "Measurement"):
  value         sweeps/s over exactly K = --steps sweeps, data resident in HBM, CUDA events on the library's stream, max over
                ranks; the timed region starts right after one throw-away sweep whose exchange lines the GPUs up
  long_run      the continuation of the same chain over >= 0.5 s of sweeps, timed on its own (clocks are sampled over both)
  e2e           sweeps/s through the public C-ABI calls with HOST (pinned) buffers: erirt_create + erirt_set_data
                (H2D + ingest) + erirt_set_state + K sweeps + erirt_get_trace/erirt_get_moments (D2H), all timed
  roofline      person-sweep kernel: algorithmic HBM bytes per launch / its mean CUDA-event duration, against the
                measured HBM copy bandwidth of MEASURED_PEAKS.json
  ess           bulk ESS per sweep of the item + structural parameters from a >= 3000-sweep run of the same chain
                (second half), ESS/s on the GPU(s) and for the CPU baseline (same ESS per sweep x CPU sweeps/s)
  sharding_check  logLike of sweeps 1..5 (f32 as benchmarked, and an f64 run): the same chain at every GPU count
  f64, crossqr, configs, c4_chains   sub-records: Float64 mode, the cell-level quantile sampler (CrossQr) at the same
                size, BASELINE configs 1-4 beside the CPU oracle, 8 independent RtIrtNull chains dealt over the GPUs
  cpu_baseline  the CPU oracle (a C restatement of the reference; Julia is not installed) on one host core, on a
                bounded sample of the persons, extrapolated linearly in nSubj
--impl reference times that same CPU restatement with all host threads (OpenMP over persons/items).
--dump-outputs DIR writes what the K timed sweeps computed (see dump_outputs) as DIR/<name>.npy; the inputs depend only on
the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, which may be read-only

N_SUBJ, N_ITEM, N_FEAT, Q_RT = 1_000_000, 100, 3, 0.85
N_BLOCKS = 8  # data is generated in 8 seeded person blocks so that every GPU count sees the same data set
SEED = 1234
METRIC = "gibbs_sweeps_per_sec"
UNIT = "sweeps/s"
WORKLOAD = "GibbsRtIrtQuantile(LatentQr) synthetic nSubj=1M nItem=100 nFeat=3 qRt=0.85 (BASELINE config 5)"
ESS_SWEEPS = 3000       # total length of the chain the ESS is taken from (second half used)
LONG_RUN_SECONDS = 0.5  # minimum device time of the long timed region


_T0 = time.perf_counter()


def log(msg):
    """Progress on stderr (the JSON line is the only thing on stdout)."""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def run_sub(name, timeout):
    """A sub-record in a child process with a hard time limit: a configuration that misbehaves at this size (it has never been the
    headline) must not take the bench line with it.  The child prints one JSON object on stdout."""
    log(f"sub-record {name} (child process, limit {timeout} s)")
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--sub", name], capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"error": f"timed out after {timeout} s"}
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            try:
                return json.loads(line)
            except Exception:
                break
    return {"error": f"rc={r.returncode}: {r.stderr[-400:]}"}


def make_config(world):
    """The `config` object of the JSON line; identical for this arm and for --impl reference at the same --gpus."""
    peer = os.environ.get("ERIRT_EXCHANGE", "peer") == "peer"
    par = "single GPU" if world <= 1 else (
        f"persons sharded over {world} GPUs, item statistics all-reduced per sweep by "
        + ("a one-shot exchange over NVLink peer memory fused into the global draw kernel" if peer else "ncclAllReduce"))
    return {"workload": WORKLOAD, "parallelism": par, "l2": "inputs (1.3 GB/sweep) larger than the 126 MB L2",
            "cuda_graph": True, "loglik_and_moments": "on"}


def true_params():
    import erirt_b200 as E
    Cond = E.setCond(nSubj=N_SUBJ, nItem=N_ITEM, nFeat=N_FEAT, qRt=Q_RT, qRa=Q_RT)
    return E.setTrueParaRtIrtLatent(Cond, rng=SEED)


def gen_block_torch(tp, block, n, device):
    """setDataRtIrtLatent(type="skew") for one block of persons, on the device, Julia column-major float64:
    returns Y^T, logT^T as (J, n) and X^T as (F, n) contiguous tensors."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(SEED * 1000 + block)
    f64 = dict(dtype=torch.float64, device=device)
    a = torch.as_tensor(tp.a, **f64)[:, None]
    b = torch.as_tensor(tp.b, **f64)[:, None]
    lam = torch.as_tensor(tp.lambda_, **f64)[:, None]
    beta = torch.as_tensor(tp.beta, **f64)
    theta = torch.randn(n, generator=g, **f64)
    X = torch.randn(N_FEAT, n, generator=g, **f64)
    # Gamma(0.5, 1) - 1 errors: Gamma(1/2) = Z^2/2
    err = 0.5 * torch.randn(n, generator=g, **f64) ** 2 - 1.0
    zeta = (beta[:N_FEAT, None] * X).sum(0) + beta[N_FEAT] * theta + err
    eta = a * (theta[None, :] - b)
    Y = (torch.rand(N_ITEM, n, generator=g, **f64) < torch.sigmoid(eta)).to(torch.float64)
    logT = lam - zeta[None, :] + torch.randn(N_ITEM, n, generator=g, **f64)
    return Y.contiguous(), logT.contiguous(), X.contiguous()


def gen_shard_torch(tp, rank, world, device):
    import torch
    per = N_SUBJ // N_BLOCKS
    blocks = range(rank * N_BLOCKS // world, (rank + 1) * N_BLOCKS // world)
    parts = [gen_block_torch(tp, bk, per, device) for bk in blocks]
    Y = torch.cat([p[0] for p in parts], dim=1).contiguous()
    T = torch.cat([p[1] for p in parts], dim=1).contiguous()
    X = torch.cat([p[2] for p in parts], dim=1).contiguous()
    return Y, T, X, blocks[0] * per, per * len(blocks)


def init_state(offset, n):
    rng = np.random.default_rng(SEED + 7)
    theta = rng.standard_normal(N_SUBJ)[offset:offset + n]
    zeta = rng.standard_normal(N_SUBJ)[offset:offset + n]
    beta = rng.standard_normal(N_FEAT + 2)
    return theta, zeta, beta


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every few milliseconds
    from a thread (ctypes releases the GIL while the library runs), so that even a 15 ms timed region gets samples;
    nvidia-smi -lms 100 is the fallback when the NVML binding is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, None
        self.thread, self.stop_flag, self.sm, self.mx, self.reasons = None, False, [], [], set()

    def _nvml_loop(self, nv, handle):
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while True:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(handle))
                for nm, bit in bits.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            if self.stop_flag:
                break
            time.sleep(0.02)  # 50 Hz: NVML calls take driver locks, a tighter loop was seen to perturb 8-GPU runs

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.idx
            handle = nv.nvmlDeviceGetHandleByIndex(phys)
            self.mx = [float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))]
            self.stop_flag = False
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if self.sm:
                out.update(sm_mhz=float(np.median(self.sm)), sm_max_mhz=float(max(self.mx)) if self.mx else None,
                           reasons=sorted(self.reasons), samples=len(self.sm), source="nvml")
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm), source="nvidia-smi")
        return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def ncu_traffic(key="dram_bytes_per_launch"):
    """dram bytes per launch of the person kernel at N=1 from the last committed ncu --set full capture (or None)."""
    p = os.path.join(ROOT, "profiles", "person_kernel_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


def bulk_ess(columns):
    """min / median rank-normalised bulk ESS (Vehtari et al. 2021) over the non-constant columns, by the engine's CUDA kernel
    (erirt_ess_rhat, csrc/diagnostics.cuh; one CTA per column)."""
    from erirt_b200.diagnostics import ess_rhat_device
    ess = np.concatenate([ess_rhat_device(arr[:, :, None])[0] for arr in columns])
    ess = ess[~np.isnan(ess)]
    return float(np.min(ess)), float(np.median(ess)), int(ess.size)


def item_struct_traces(eng, first, n, qw):
    N, J = eng.N, eng.J
    has_rt = eng.model != 0
    cols = [eng.get_trace("ra", N, 2 * J)[first:first + n, :, 0]]
    if has_rt:
        cols.append(eng.get_trace("rt", N, 2 * J)[first:first + n, :, 0])
    cols.append(eng.get_trace("qr", 0, qw)[first:first + n, :, 0])
    return cols


DUMP_PERSONS = 1 << 18  # person-level outputs are written for this many persons (fixed sample drawn with SEED)


def dump_outputs(eng, out_dir, last, world, rank):
    """What a caller of the timed path receives after its last sweep (api.sample's MCMC.Para and Post), as out_dir/<name>.npy in
    float64: theta and zeta (erirt_get_state), the running mean and SD of theta, zeta and nu (erirt_get_moments), and a, b, lambda,
    sigma2, beta, Sigma_p and logLike from trace row `last`.  The eight person-level arrays are restricted to the same seeded sample
    of DUMP_PERSONS persons (ascending ids), so that everything stays near 17 MB.  The item statistics are summed with atomics, so
    two runs of one build agree only up to that rounding as the chain carries it forward (on a B200 in f32: logLike of sweep 1 within
    1e-10 relative, person draws within 0.1 after 26 sweeps).  Collective when world > 1."""
    from erirt_b200 import distributed as D
    J = N_ITEM
    person = {"theta": eng.get_state("theta"), "zeta": eng.get_state("zeta")}
    for f in ("theta", "zeta", "nu"):
        person[f + "_mean"], person[f + "_sd"] = eng.get_moments(f)
    if world > 1:
        person = {k: D.gather_person_vector(v, N_SUBJ) for k, v in person.items()}
    if rank != 0:
        return
    idx = np.sort(np.random.default_rng(SEED).choice(N_SUBJ, DUMP_PERSONS, replace=False))
    out = {k: v[idx] for k, v in person.items()}
    ra = eng.get_trace("ra", eng.N, 2 * J)[last, :, 0]
    rt = eng.get_trace("rt", eng.N, 2 * J)[last, :, 0]
    qr = eng.get_trace("qr", 0, N_FEAT + 6)[last, :, 0]
    out.update({"a": ra[:J], "b": ra[J:], "lambda": rt[:J], "sigma2": rt[J:], "beta": qr[:N_FEAT + 2],
                "Sigma_p": qr[N_FEAT + 2:].reshape(2, 2, order="F"), "logLike": eng.get_trace("logLike")[last, :, 0]})
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(v, dtype=np.float64))
    log(f"outputs of sweep {last + 1} written to {out_dir}")


def cpu_oracle_rate(tp, n_sample, n_sweeps, nthreads, warm=1):
    """sweeps/s of the CPU restatement on the first n_sample persons of block 0 (host-generated, same
    distributions), extrapolated linearly to N_SUBJ persons."""
    import copy
    import erirt_b200 as E
    from oracle import oracle_py as O
    Cond = E.setCond(nSubj=n_sample, nItem=N_ITEM, nFeat=N_FEAT, qRt=Q_RT)
    tpc = copy.deepcopy(tp)
    D = E.setDataRtIrtLatent(Cond, tpc, type="skew", rng=SEED)
    cfg = O.make_cfg("RtIrtLatentQr", n_sample, N_ITEM, N_FEAT, qRt=Q_RT, seed=SEED, nthreads=nthreads)
    theta, zeta, beta = init_state(0, n_sample)
    init = dict(theta=theta, zeta=zeta, beta=beta, a=np.ones(N_ITEM), b=np.zeros(N_ITEM), lambda_=np.zeros(N_ITEM),
                sigma2=np.ones(N_ITEM), Sigma=np.eye(2).ravel())
    if warm:
        O.sample(cfg, D.Y, D.logT, D.X, init, warm, person_trace=False, qr_skip_nu=True)
    t0 = time.perf_counter()
    O.sample(cfg, D.Y, D.logT, D.X, init, n_sweeps, person_trace=False, qr_skip_nu=True)
    dt = time.perf_counter() - t0
    return (n_sweeps / dt) * (n_sample / N_SUBJ), dt


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The Julia package cannot
    run here (no julia binary), so this is the oracle port with all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as O
    O.build()
    tp = true_params()
    cores = os.cpu_count() or 1
    total = args.steps + args.warmup
    # calibrate so that the whole run stays within ~2 minutes
    rate, _ = cpu_oracle_rate(tp, 2000, 2, cores, warm=1)
    per_sweep_full = 1.0 / rate
    budget = 100.0 / max(total, 1)
    n_sample = int(min(N_SUBJ, max(2000, N_SUBJ * budget / per_sweep_full)))
    n_sample -= n_sample % 8
    value, dt = cpu_oracle_rate(tp, n_sample, args.steps, cores, warm=args.warmup)
    sample = (f"oracle (C restatement of Draw.pl.jl, not Julia) with {cores} OpenMP threads on the first {n_sample} persons x {N_ITEM} items, "
              f"{args.steps} sweeps in {dt:.1f} s, sweeps/s scaled by {n_sample}/{N_SUBJ} (cost is linear in persons)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": make_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# sub-records (single GPU only): Float64 mode, CrossQr at C5 size, BASELINE configs 1-4 beside the CPU oracle
# ------------------------------------------------------------------------------------------------------------------
def roofline_record(eng_stats, kernel_ms, kernel_name, launches):
    peak, which = measured_peak()
    b = eng_stats["bytes_per_sweep"]
    achieved = b / (kernel_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "peak_source": which, "unit": "GB/s",
            "frac": achieved / peak, "algorithmic_bytes_per_launch": b, "kernel_ms": kernel_ms, "launches_timed": launches}


def sub_f64(E, local):
    """The benchmarked sampler in Float64 (the reference's precision): 25 B per cell."""
    import torch
    dY, dT, dX, _, n_local = gen_shard_torch(true_params(), 0, 1, torch.device("cuda", local))
    theta0, zeta0, beta0 = init_state(0, n_local)
    out = {}
    for timed in (False, True):
        eng = E.Engine("RtIrtQuantile", n_local, N_ITEM, N_FEAT, n_iter=64, n_chain=1, n_burnin=0, q_rt=Q_RT, cov2one=False, dtype="f64",
                       seed=SEED, person_trace=False, device=local, use_graph=not timed, time_kernels=timed)
        eng.set_data_device(dY.data_ptr(), n_local, dT.data_ptr(), n_local, dX.data_ptr(), n_local)
        eng.set_state(theta=theta0, zeta=zeta0, beta=beta0)
        eng.sample(4)
        eng.sample(20)
        st = eng.stats()
        if not timed:
            out.update(value=20 / (st["last_sample_ms"] / 1e3), unit=UNIT, ms_per_step=st["last_sample_ms"] / 20, sweeps=20, dtype="f64")
        else:
            out["roofline"] = roofline_record(st, st["person_kernel_ms"], "person_sweep_kernel<double>", 20)
        eng.close()
    return out


def sub_crossqr(E, local):
    """GibbsRtIrtCrossQr (cell-level quantile weights nu_ij, src/GibbsRtIrtCross.pl.jl:265-325) at 1M x 100, q = 0.85, data from
    setDataRtIrtCross(type="skew") generated on the device; two person launches per sweep (K_a, K_b): 29 / 57 B per cell."""
    Cond = E.setCond(nSubj=N_SUBJ, nItem=N_ITEM, nFeat=0, qRt=Q_RT)
    tp = E.setTrueParaRtIrtCross(Cond, rng=SEED)
    rng = np.random.default_rng(SEED + 21)
    theta, zeta = rng.standard_normal(N_SUBJ), rng.standard_normal(N_SUBJ)
    out = {"workload": "GibbsRtIrtCrossQr synthetic nSubj=1M nItem=100 qRt=0.85, setDataRtIrtCross(type=skew)"}
    for dtype in ("f32", "f64"):
        rec = {}
        for timed in (False, True):
            eng = E.Engine("RtIrtCrossQr", N_SUBJ, N_ITEM, 0, n_iter=64, n_chain=1, n_burnin=0, q_rt=Q_RT, cov2one=True, dtype=dtype,
                           seed=SEED, person_trace=False, device=local, use_graph=not timed, time_kernels=timed)
            eng.generate_data(theta, tp.a, tp.b, zeta, tp.lambda_, tp.sigma2t, tp.rho, None, error="skew", seed=SEED)
            eng.set_state(theta=rng.standard_normal(N_SUBJ), zeta=rng.standard_normal(N_SUBJ), rho=np.zeros(N_ITEM))
            n = 12
            eng.sample(3)
            eng.sample(n)
            st = eng.stats()
            if not timed:
                b = st["bytes_per_sweep"]
                peak, which = measured_peak()
                ms = st["last_sample_ms"] / n
                rec.update(value=1e3 / ms, unit=UNIT, ms_per_step=ms, sweeps=n,
                           roofline={"bound": "hbm", "kernel": "person_sweep_kernel<FAM=1> K_a + K_b (whole sweep)", "achieved": b / (ms * 1e-3) / 1e9,
                                     "peak": peak, "peak_source": which, "unit": "GB/s", "frac": b / (ms * 1e-3) / 1e9 / peak,
                                     "algorithmic_bytes_per_sweep": b})
            else:
                rec["k_b_kernel_ms"] = st["person_kernel_ms"]
            ll = eng.get_trace("logLike")[:n + 3, 0, 0]
            assert np.all(np.isfinite(ll)), "CrossQr logLike not finite"
            eng.close()
        out[dtype] = rec
    return out


def _time_engine(E, model, Data, N, J, F, n_iter, n_chain, dtype, init, local, q_rt=0.5, cov2one=True, warm=50):
    eng = E.Engine(model, N, J, F, n_iter=n_iter, n_chain=n_chain, n_burnin=0, q_rt=q_rt, cov2one=cov2one, dtype=dtype, seed=SEED,
                   person_trace=False, device=local, use_graph=True)
    eng.set_data(Data.Y, None if model == "MlIrt" else Data.logT, Data.X if F > 0 else None)
    eng.set_state(**init)
    total = n_iter * n_chain
    eng.sample(warm)
    eng.sample(total - warm)
    ms = eng.stats()["last_sample_ms"] / (total - warm)
    eng.close()
    return 1e3 / ms


def _time_oracle(model, Data, N, J, F, init, n_sweeps, q_rt=0.5, cov2one=None):
    from oracle import oracle_py as O
    cfg = O.make_cfg(model, N, J, F, qRt=q_rt, seed=SEED, nthreads=1, cov2one=cov2one)
    logT = None if model == "MlIrt" else Data.logT
    O.sample(cfg, Data.Y, logT, Data.X, init, 1, person_trace=False, qr_skip_nu=True)
    t0 = time.perf_counter()
    O.sample(cfg, Data.Y, logT, Data.X, init, n_sweeps, person_trace=False, qr_skip_nu=True)
    return n_sweeps / (time.perf_counter() - t0)


def sub_configs(E, local):
    """BASELINE configs 1-4 (SURVEY 8d): sweeps/s on one GPU (f32 and f64, CUDA-graph replay, everything on) beside the CPU oracle on
    one core.  These problems are launch / latency bound (their working set is L2- or SM-resident): no roofline fraction applies."""
    rng = np.random.default_rng(SEED + 31)
    out = {}

    def rec(name, model, N, J, F, n_iter, n_chain, Data, init, cpu_sweeps, q_rt=0.5, cov2one=True):
        r = {"workload": name, "n_subj": N, "n_item": J, "n_feat": F, "n_chain": n_chain}
        for dt in ("f32", "f64"):
            r[f"gpu_{dt}_sweeps_per_s"] = _time_engine(E, model, Data, N, J, F, n_iter, n_chain, dt, init, local, q_rt, cov2one)
        oinit = dict(a=np.ones(J), b=np.zeros(J), lambda_=np.zeros(J), sigma2=np.ones(J), Sigma=np.eye(2).ravel())
        oinit.update({k.rstrip("_"): v for k, v in init.items()})
        r["cpu_oracle_sweeps_per_s"] = _time_oracle(model, Data, N, J, F, oinit, cpu_sweeps, q_rt, cov2one)
        r["cpu_cores"] = 1
        out[name.split(":")[0]] = r

    # C1: GibbsMlIrt README simulation, 1000 x 15, single chain
    Cond = E.setCond(nSubj=1000, nItem=15, nFeat=3, nIter=3000, nChain=1)
    tp = E.setTrueParaMlIrt(Cond, rng=SEED)
    D = E.setDataMlIrt(Cond, tp, rng=SEED)
    rec("C1: GibbsMlIrt README simulation 1000x15 single chain", "MlIrt", 1000, 15, 3, 3000, 1, D,
        dict(theta=rng.standard_normal(1000), beta=rng.standard_normal(4)), 300)
    # C2: GibbsRtIrt 10k x 30, nChain = 3 (the reference's interleaved chains)
    Cond = E.setCond(nSubj=10_000, nItem=30, nFeat=3, nIter=1000, nChain=3)
    tp = E.setTrueParaRtIrt(Cond, rng=SEED)
    D = E.setDataRtIrt(Cond, tp, rng=SEED)
    rec("C2: GibbsRtIrt 10k x 30 nChain=3", "RtIrt", 10_000, 30, 3, 1000, 3, D,
        dict(theta=rng.standard_normal(10_000), zeta=rng.standard_normal(10_000), beta=rng.standard_normal(8)), 20)
    # C3: GibbsRtIrtQuantile q = 0.85 on TIMSS-shaped data 631 x 14, F = 10
    Cond = E.setCond(nSubj=631, nItem=14, nFeat=10, nIter=1000, nChain=3, qRt=0.85)
    tp = E.setTrueParaRtIrtLatent(Cond, rng=SEED)
    D = E.setDataRtIrtLatent(Cond, tp, type="norm", rng=SEED)
    rec("C3: GibbsRtIrtQuantile q=0.85 TIMSS-shaped 631x14 F=10 nChain=3", "RtIrtLatentQr", 631, 14, 10, 1000, 3, D,
        dict(theta=rng.standard_normal(631), zeta=rng.standard_normal(631), beta=rng.standard_normal(12)), 300, q_rt=0.85, cov2one=False)
    # C4: GibbsRtIrtNull 100k x 40, one of the 8 chains (the 8-chain run over the GPUs is the c4_chains record)
    Cond = E.setCond(nSubj=100_000, nItem=40, nFeat=0, nIter=1000, nChain=1)
    tp = E.setTrueParaRtIrt(Cond, rng=SEED)
    D = E.setDataRtIrtNull(Cond, tp, rng=SEED)
    rec("C4: GibbsRtIrtNull 100k x 40 one chain", "RtIrtNull", 100_000, 40, 0, 1000, 1, D,
        dict(theta=rng.standard_normal(100_000), zeta=rng.standard_normal(100_000)), 3)
    return out


def c4_chains(E, rank, world, local, n_chains=8, n_iter=1000):
    """BASELINE configs[3]: 8 independent GibbsRtIrtNull chains at 100k x 40 dealt over the ranks (chain c on rank c mod world, the
    chains of a rank one after the other), no collective while sampling; chains x sweeps per second (max over ranks of the
    device time) and the cross-chain split R-hat of the item parameters from the second half of the n_iter sweeps."""
    import torch
    from erirt_b200 import distributed as D
    from erirt_b200.diagnostics import ess_rhat_device
    N, J = 100_000, 40
    Cond = E.setCond(nSubj=N, nItem=J, nFeat=0, nIter=n_iter, nChain=1)
    tp = E.setTrueParaRtIrt(Cond, rng=SEED)
    Data = E.setDataRtIrtNull(Cond, tp, rng=SEED)
    mine = D.chain_assignment(n_chains, world, rank)
    ms_total, traces = 0.0, {}
    for c in mine:
        rng = np.random.default_rng(SEED + 1000 + c)
        eng = E.Engine("RtIrtNull", N, J, 0, n_iter=n_iter, n_chain=1, n_burnin=n_iter // 2, dtype="f32", seed=SEED, chain=c,
                       person_trace=False, device=local, use_graph=True)
        eng.set_data(Data.Y, Data.logT, None)
        eng.set_state(theta=rng.standard_normal(N), zeta=rng.standard_normal(N))
        eng.sample(n_iter)
        ms_total += eng.stats()["last_sample_ms"]
        traces[c] = np.concatenate([eng.get_trace("ra", N, 2 * J)[n_iter // 2:, :, 0], eng.get_trace("rt", N, 2 * J)[n_iter // 2:, :, 0]], axis=1)
        eng.close()
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms_total], dtype=torch.float64, device=torch.device("cuda", local))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        parts = [None] * world
        dist.all_gather_object(parts, traces)
        traces = {c: v for part in parts for c, v in part.items()}
    if rank != 0:
        return None
    arr = np.stack([traces[c] for c in range(n_chains)], axis=2)  # [iter, param, chain]
    rhat = ess_rhat_device(arr, device=local)[1]  # CUDA kernel, one CTA per column
    return {"workload": f"{n_chains} independent GibbsRtIrtNull chains 100k x 40, {n_iter} sweeps each, chain c on rank c mod {world}",
            "value": n_chains * n_iter / (ms_total / 1e3), "unit": "chain-sweeps/s", "chains": n_chains, "sweeps_per_chain": n_iter,
            "seconds_max_over_ranks": ms_total / 1e3, "rhat_max": float(np.nanmax(rhat)), "rhat_median": float(np.nanmedian(rhat)),
            "rhat_params": "a, b, lambda, sigma2 (160 columns), split R-hat over the 8 chains, second half of each chain"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="erirt_b200", choices=["erirt_b200", "reference"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-y", choices=["u8", "f64"], default="u8", help="host type of Y in the end-to-end pass (Julia Matrix{Bool} or Float64)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sub-records (f64, crossqr, configs, c4_chains, ess)")
    ap.add_argument("--short", action="store_true", help="profiling run: timed sweeps only, no e2e / cpu / roofline / sub-record passes")
    ap.add_argument("--sub", default=None, choices=["f64", "crossqr", "configs"], help="(internal) run one sub-record and print it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed sweeps computed (state, moments, last trace row) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)
    if args.sub:
        import torch
        import erirt_b200 as E
        torch.cuda.set_device(0)
        rec = {"f64": sub_f64, "crossqr": sub_crossqr, "configs": sub_configs}[args.sub](E, 0)
        print(json.dumps(rec), flush=True)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import erirt_b200 as E
    from erirt_b200 import distributed as D

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    assert N_BLOCKS % world == 0, "GPU count must divide 8"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    extras = not (args.short or args.no_extras)

    tp = true_params()
    dY, dT, dX, offset, n_local = gen_shard_torch(tp, rank, world, dev)
    theta0, zeta0, beta0 = init_state(offset, n_local)
    K, W = args.steps, args.warmup
    qw = N_FEAT + 2 + 4

    def make_engine(time_kernels=False, use_graph=True, dtype=None, n_iter=None):
        eng = E.Engine("RtIrtQuantile", n_local, N_ITEM, N_FEAT, n_iter=n_iter or (K + W + 8), n_chain=1, n_burnin=0, q_rt=Q_RT,
                       cov2one=False, dtype=dtype or args.dtype, seed=SEED, person_trace=False, device=local, use_graph=use_graph,
                       n_subj_total=N_SUBJ, subj_offset=offset, time_kernels=time_kernels)
        if world > 1:
            peer = os.environ.get("ERIRT_EXCHANGE", "peer") == "peer"
            sh, _ = D.make_shard(N_SUBJ, nccl=not peer)  # NCCL mode: a fresh id per communicator
            eng.comm_init(sh[0], sh[1], sh[2])
            if peer:
                D.attach_peers(eng)  # one-shot exchange over NVLink peer memory fused into the global draw kernel; no NCCL at all
        return eng

    def close_engine(e):
        if world > 1:
            D.close_sharded(e)  # unmap the peers' exchange buffers on every rank before anybody frees its own
        else:
            e.close()

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    log("data generated; value / long run / ESS chain")
    # ---------------- device-resident throughput ("value"), the long run, the ESS chain ----------------
    cap = max(ESS_SWEEPS, 2 * (K + W)) + 4096 if (extras or not args.short) else K + W + 8  # the long run needs room too
    eng = make_engine(n_iter=cap)
    eng.set_data_device(dY.data_ptr(), n_local, dT.data_ptr(), n_local, dX.data_ptr(), n_local)
    eng.set_state(theta=theta0, zeta=zeta0, beta=beta0)
    eng.sample(W)
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    eng.sample(1)  # throw-away sweep: its exchange is the device-side rendezvous of the ranks (the host barrier leaves them up to ~1 ms apart)
    eng.sample(K)
    ms = max_over_ranks(eng.stats()["last_sample_ms"])
    done = W + 1 + K
    if args.dump_outputs:
        dump_outputs(eng, args.dump_outputs, done - 1, world, rank)
    long_run = None
    if not args.short:
        n_long = int(max(1, min(cap - done - 8, max(K, math.ceil(LONG_RUN_SECONDS * 1e3 / (ms / K))))))
        if world > 1:
            eng.sample(1)
            done += 1
        eng.sample(n_long)
        ms_long = max_over_ranks(eng.stats()["last_sample_ms"])
        done += n_long
        long_run = {"sweeps": n_long, "ms_per_step": ms_long / n_long, "value": n_long / (ms_long / 1e3), "unit": UNIT,
                    "note": f"the same chain continued for >= {LONG_RUN_SECONDS} s of device time, CUDA events, max over ranks"}
    barrier()
    clk = clocks.stop()
    st = eng.stats()
    value = K / (ms / 1000.0)
    ll_first = [float(v) for v in eng.get_trace("logLike")[:5, 0, 0]] if rank == 0 else None
    log(f"value {value:.1f} sweeps/s ({ms / K:.4f} ms/sweep)" + (f", long run {long_run['ms_per_step']:.4f} ms/sweep over {long_run['sweeps']}" if long_run else ""))
    ess = None
    if extras:
        if done < ESS_SWEEPS:
            eng.sample(ESS_SWEEPS - done)
            done = ESS_SWEEPS
        if rank == 0:
            try:
                half = done // 2
                e_min, e_med, n_par = bulk_ess(item_struct_traces(eng, half, done - half, qw))
                ess = {"chain_sweeps": done, "used_sweeps": done - half, "params": n_par, "min": e_min, "median": e_med,
                       "per_sweep_min": e_min / (done - half), "per_sweep_median": e_med / (done - half),
                       "per_sec_min": e_min / (done - half) * value, "per_sec_median": e_med / (done - half) * value,
                       "estimator": "rank-normalised split bulk ESS (Vehtari et al. 2021) of a, b, lambda, sigma2, beta, Sigma_p over the second half of the chain"}
            except Exception as ex:
                ess = {"error": str(ex)}
    close_engine(eng)

    log("ESS done; f64 sharding check")
    # ---------------- sharding check in f64: logLike of sweeps 1..5 of the same chain at every GPU count ----------------
    ll64 = None
    if extras:
        e64 = make_engine(dtype="f64", n_iter=8)
        e64.set_data_device(dY.data_ptr(), n_local, dT.data_ptr(), n_local, dX.data_ptr(), n_local)
        e64.set_state(theta=theta0, zeta=zeta0, beta=beta0)
        e64.sample(5)
        if rank == 0:
            ll64 = [float(v) for v in e64.get_trace("logLike")[:5, 0, 0]]
        close_engine(e64)

    log("roofline pass")
    # ---------------- roofline of the person kernel (plain launches bracketed by CUDA events) ----------------
    roofline = None
    if not args.short:
        engk = make_engine(time_kernels=True, use_graph=False)
        engk.set_data_device(dY.data_ptr(), n_local, dT.data_ptr(), n_local, dX.data_ptr(), n_local)
        engk.set_state(theta=theta0, zeta=zeta0, beta=beta0)
        engk.sample(min(W, 10))
        barrier()
        kk = min(K, 100)
        engk.sample(kk)
        sk = engk.stats()
        pk_ms = max_over_ranks(sk["person_kernel_ms"])
        roofline = roofline_record(sk, pk_ms, "person_sweep_fast_kernel" if args.dtype == "f32" else "person_sweep_kernel", kk)
        # dram bytes of one launch come from the committed ncu --set full capture at N = 1 (profiles/person_kernel_traffic.json): quoted
        # for the single-GPU line only, where a launch processes the same 1M x 100 cells as the capture
        roofline["traffic"] = ncu_traffic() if world == 1 else None
        roofline["traffic_source"] = "profiles/person_kernel_traffic.json (ncu --set full of this kernel at N=1; not re-measured by this run)" if world == 1 else None
        roofline["pg_deferred_frac"] = sk["pg_deferred_frac"]
        roofline["ideal_kernel_ms_at_this_n"] = None
        close_engine(engk)

    # ---------------- sub-records that only need one GPU ----------------
    f64_rec = crossqr_rec = configs_rec = None

    log("e2e pass")
    # ---------------- end to end through the C ABI with host buffers ("e2e") ----------------
    e2e = None
    if not args.no_e2e and not args.short:
        # the host holds what the reference's InputData holds: Y as Julia's Matrix{Bool} (one byte per response, `rand.(BernoulliLogit…)`
        # src/SimTools.jl:165; --e2e-y f64 passes a Float64 Y instead), logT and X as Float64; all column-major, pinned
        y8 = args.e2e_y == "u8"
        hY = torch.empty(dY.shape, dtype=torch.uint8 if y8 else torch.float64, pin_memory=True).copy_(dY)
        hT = torch.empty(dT.shape, dtype=torch.float64, pin_memory=True).copy_(dT)
        hX = torch.empty(dX.shape, dtype=torch.float64, pin_memory=True).copy_(dX)
        hM = torch.empty((3, 2, n_local), dtype=torch.float64, pin_memory=True)  # Post.mean / SD of theta, zeta, nu land here
        hMn = hM.numpy()
        del dY, dT, dX
        torch.cuda.empty_cache()
        barrier()
        t0 = time.perf_counter()
        enge = make_engine()
        t1 = time.perf_counter()
        from erirt_b200._lib import check
        set_data = enge.lib.erirt_set_data_y8 if y8 else enge.lib.erirt_set_data
        check(set_data(enge.h, hY.data_ptr(), n_local, hT.data_ptr(), n_local, hX.data_ptr(), n_local))
        enge.set_state(theta=theta0, zeta=zeta0, beta=beta0)
        t2 = time.perf_counter()
        enge.sample(K)
        t3 = time.perf_counter()
        tr_a = enge.get_trace("ra", n_local, 2 * N_ITEM)
        tr_t = enge.get_trace("rt", n_local, 2 * N_ITEM)
        tr_q = enge.get_trace("qr", 0, qw)
        tr_l = enge.get_trace("logLike")
        moms = [enge.get_moments(f, out=(hMn[k, 0], hMn[k, 1])) for k, f in enumerate(("theta", "zeta", "nu"))]
        t4 = time.perf_counter()
        close_engine(enge)  # erirt_destroy is part of the call a user makes (the Julia shim destroys the handle inside sample!)
        t5 = time.perf_counter()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        h2d = hY.numel() * hY.element_size() + (hT.numel() + hX.numel()) * 8 + (2 * n_local + N_FEAT + 2) * 8
        d2h = K * (tr_a.shape[1] + tr_t.shape[1] + tr_q.shape[1] + 1) * 8 + 3 * 2 * n_local * 8
        assert np.all(np.isfinite(tr_l[:K])) and np.all(np.isfinite(moms[0][0]))
        e2e = {"value": K / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d * world / K), "d2h_bytes_per_step": int(d2h * world / K),
               "seconds": dt, "parts_ms_rank0": {"create": (t1 - t0) * 1e3, "set_data_and_state": (t2 - t1) * 1e3, "sample": (t3 - t2) * 1e3, "read_back": (t4 - t3) * 1e3, "destroy": (t5 - t4) * 1e3},
               "note": "erirt_create + " + ("erirt_set_data_y8 (pinned host: Y as Matrix{Bool} bytes, logT/X f64" if y8 else "erirt_set_data (pinned host f64")
                                     + "; chunked H2D + ingest) + erirt_set_state + K sweeps + "
                                     "erirt_get_trace/erirt_get_moments (D2H into pinned buffers) + erirt_destroy; bytes are totals of the call divided by K"}
        del hY, hT, hX
    else:
        del dY, dT, dX
        torch.cuda.empty_cache()
        hMn = np.empty((3, 2, n_local))

    log("e2e with device-generated data")
    # ---------------- the same call with the N x J data generated on the device (informational: no N x J upload) ----------------
    e2e_gen = None
    if not args.no_e2e and not args.short:
        rng = np.random.default_rng(SEED + 11)
        th_all = rng.standard_normal(N_SUBJ)
        X_all = rng.standard_normal((N_SUBJ, N_FEAT))
        ze_all = np.column_stack([X_all, th_all]) @ tp.beta + (0.5 * rng.standard_normal(N_SUBJ) ** 2 - 1.0)  # setDataRtIrtLatent(type="skew")
        sl = slice(offset, offset + n_local)
        th_g, ze_g, X_g = th_all[sl].copy(), ze_all[sl].copy(), np.asfortranarray(X_all[sl])
        barrier()
        t0 = time.perf_counter()
        engg = make_engine()
        engg.generate_data(th_g, tp.a, tp.b, ze_g, tp.lambda_, None, None, X_g, error="unit", seed=SEED)
        engg.set_state(theta=theta0, zeta=zeta0, beta=beta0)
        engg.sample(K)
        tr_g = [engg.get_trace("ra", n_local, 2 * N_ITEM), engg.get_trace("rt", n_local, 2 * N_ITEM), engg.get_trace("qr", 0, qw), engg.get_trace("logLike")]
        moms_g = [engg.get_moments(f, out=(hMn[k, 0], hMn[k, 1])) for k, f in enumerate(("theta", "zeta", "nu"))]
        close_engine(engg)
        barrier()
        dtg = max_over_ranks(time.perf_counter() - t0)
        assert np.all(np.isfinite(tr_g[3][:K])) and np.all(np.isfinite(moms_g[0][0]))
        e2e_gen = {"value": K / dtg, "unit": UNIT, "seconds": dtg, "h2d_bytes_per_step": int((2 + N_FEAT) * n_local * 8 * world / K),
                   "note": "erirt_create + erirt_generate_data (person-level theta, zeta, X from the host; responses and log-times generated "
                           "on the device) + erirt_set_state + K sweeps + read-back + erirt_destroy"}

    chains_rec = None
    if extras:
        log("c4_chains: 8 independent RtIrtNull chains")
        try:
            chains_rec = c4_chains(E, rank, world, local)
        except Exception as ex:
            chains_rec = {"error": str(ex)}
    if extras and world == 1:
        torch.cuda.empty_cache()
        f64_rec = run_sub("f64", 180)
        configs_rec = run_sub("configs", 240)
        crossqr_rec = run_sub("crossqr", 240)

    log("cpu baseline")
    # ---------------- CPU baseline beside it (rank 0, single GPU run only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and not args.short:
        try:
            n_sample = 40000
            v, dtc = cpu_oracle_rate(tp, n_sample, 8, 1, warm=1)
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"oracle (C restatement of Draw.pl.jl; the Julia reference cannot run here) on 1 core of {os.cpu_count()}, "
                             f"first {n_sample} persons x {N_ITEM} items, 8 sweeps in {dtc:.1f} s, scaled by {n_sample}/{N_SUBJ}"}
            if ess and "per_sweep_min" in ess:
                cpu["ess_per_sec_min"] = ess["per_sweep_min"] * v
                cpu["ess_per_sec_median"] = ess["per_sweep_median"] * v
                cpu["ess_note"] = "ESS per sweep is a property of the scan (measured once, on the GPU chain) x CPU sweeps/s"
        except Exception as ex:  # the bench line must still be printed
            cpu = {"value": None, "unit": UNIT, "cores": 1, "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "timed_sweeps": K,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": args.dtype, "data": "synthetic", "config": make_config(world),
                "clocks": clk, "gpu_launches": 2 * K, "long_run": long_run, "e2e": e2e, "e2e_device_generated_data": e2e_gen,
                "roofline": roofline, "cpu_baseline": cpu, "ess": ess,
                "sharding_check": {"loglike_sweeps_1_5_" + args.dtype: ll_first, "loglike_sweeps_1_5_f64": ll64,
                                   "note": "the same chain (seed, data, initial state) at every GPU count: Philox counters use global person ids, "
                                           "so the values agree across N up to the summation order of the statistics"},
                "f64": f64_rec, "crossqr": crossqr_rec, "configs": configs_rec, "c4_chains": chains_rec,
                "bytes_per_sweep": st["bytes_per_sweep"] * world}
        if roofline is not None:
            roofline["ideal_kernel_ms_at_this_n"] = ncu_traffic("kernel_ms_n1") / world if ncu_traffic("kernel_ms_n1") else None
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
