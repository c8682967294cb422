"""Replica batches (erirt_create_batch, DESIGN.md 6.6) against the same replicas run one after another.

Prints one JSON line:
  grid: RtIrt, J = 15, F = 3, for dtype in {f32, f64}, N in {250, 500, 1000}, B in {1, 8, 32, 100}: replica-sweeps/s of one batch of
        B replicas, and of B standalone engines sampled one after another over the same sweeps (device time of erirt_sample, CUDA
        events, summed over the engines), and their ratio;
  runSimulation: wall time of simtools.runSimulation (RtIrt, nRep = 100, nIter = 2000, nChain = 3, N = 1000, J = 15, F = 3, f64)
        with batch=100 against batch=None;
and the card's name and power limit, read in the same run.
Usage: python tools/bench_batch.py [--sweeps 320] [--skip-sim]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return name, pl


def problem(N, seed):
    from helpers import make_problem
    return make_problem("RtIrt", N, 15, 3, seed=seed)


def engine(E, pb, dtype, n_iter, seed, n_batch=1):
    return E.Engine("RtIrt", pb["N"], 15, 3, n_iter=n_iter, n_chain=1, n_burnin=n_iter // 2, q_rt=pb["q"], dtype=dtype, seed=seed,
                    person_trace=False, use_graph=True, n_batch=n_batch)


def init(pb):
    i = pb["init"]
    return dict(theta=i["theta"], zeta=i["zeta"], a=i["a"], b=i["b"], lambda_=i["lambda_"], sigma2=i["sigma2"], Sigma=i["Sigma"],
                beta=i["beta"][: pb["nb"]])


def grid_point(E, dtype, N, B, sweeps, warm=32):
    pbs = [problem(N, 100 + r) for r in range(B)]
    n_iter = warm + sweeps
    # batch
    eng = engine(E, pbs[0], dtype, n_iter, 1, n_batch=B)
    eng.set_data(*(np.concatenate([p[k] for p in pbs], axis=0) for k in ("Y", "logT", "X")))  # replicas stacked along the rows
    inits = [init(p) for p in pbs]
    eng.set_state(**{k: [i[k] for i in inits] for k in inits[0]})
    eng.sample(warm)
    eng.sample(sweeps)
    t_batch = eng.stats()["last_sample_ms"] * 1e-3
    eng.close()
    # the same replicas one after another
    t_seq = 0.0
    for r, pb in enumerate(pbs):
        one = engine(E, pb, dtype, n_iter, 1 + r)
        one.set_data(pb["Y"], pb["logT"], pb["X"])
        one.set_state(**init(pb))
        one.sample(warm)
        one.sample(sweeps)
        t_seq += one.stats()["last_sample_ms"] * 1e-3
        one.close()
    rb, rs = B * sweeps / t_batch, B * sweeps / t_seq
    return dict(dtype=dtype, N=N, B=B, sweeps=sweeps, batch_replica_sweeps_per_s=round(rb, 1), sequential_replica_sweeps_per_s=round(rs, 1),
                speedup=round(rb / rs, 2))


def run_simulation(batch):
    from erirt_b200 import api, simtools, simulate, structs
    C = structs.setCond(nSubj=1000, nItem=15, nFeat=3, nIter=2000, nChain=3, nRep=100)
    tp = simulate.setTrueParaRtIrt(C, rng=7)
    t0 = time.perf_counter()
    simtools.runSimulation(C, tp, funcData=simulate.setDataRtIrt, funcGibbs=api.GibbsRtIrt, seed=11, dtype="f64", person_trace=False,
                           batch=batch)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=320)
    ap.add_argument("--skip-sim", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_batch.py needs a CUDA device")
    import erirt_b200 as E
    name, power = card()
    grid = [grid_point(E, dt, N, B, args.sweeps) for dt in ("f32", "f64") for N in (250, 500, 1000) for B in (1, 8, 32, 100)]
    out = dict(card=name, power_limit=power, model="RtIrt", J=15, F=3, grid=grid)
    if not args.skip_sim:
        run_simulation(2)  # warm-up: module load, graph capture paths
        tb, ts = run_simulation(100), run_simulation(None)
        out["runSimulation"] = dict(nRep=100, nIter=2000, nChain=3, N=1000, dtype="f64", batch100_s=round(tb, 2), sequential_s=round(ts, 2),
                                    speedup=round(ts / tb, 2))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
