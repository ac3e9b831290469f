#!/usr/bin/env python
"""Energy mover's distance: gnn_jet_autoencoder_b200.anomaly.emd (one gj_emd launch for the batch) against the per-jet float64
linear program (scipy.optimize.linprog, HiGHS) that a host implementation solves jet by jet, timed on a subset and extrapolated.

Inputs: two independent synthetic_jets batches (JetNet-shaped [pt, eta, phi], zero padded), default options (R = 1, beta = 1,
norm = False).  GPU box: python tools/emd_bench.py [--out result.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for path in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, path)
import numpy as np
import torch

import emd_oracle as O
from gnn_jet_autoencoder_b200 import anomaly
from gnn_jet_autoencoder_b200.trainer import synthetic_jets


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def time_device(p, q, reps):
    anomaly.emd(p, q)                                     # warm-up: module load, shared-memory attribute
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        out = anomaly.emd(p, q)
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / reps, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    name, power = gpu_info()
    results = []
    for N, B, n_lp in ((30, 65536, 64), (150, 2048, 4)):
        p_np, q_np = synthetic_jets(B, N, seed=11), synthetic_jets(B, N, seed=12)
        p, q = torch.from_numpy(p_np).cuda(), torch.from_numpy(q_np).cuda()
        ms, out = time_device(p, q, args.reps)
        t0 = time.perf_counter()
        ref = np.array([O.emd_lp(p_np[b], q_np[b])[0] for b in range(n_lp)])
        lp_s = (time.perf_counter() - t0) / n_lp
        got = out[:n_lp].cpu().numpy()
        r = dict(N=N, B=B, emd_ms=round(ms, 3), emd_jets_per_s=round(B / ms * 1e3), linprog_jets_timed=n_lp,
                 linprog_ms_per_jet=round(lp_s * 1e3, 2), linprog_batch_s_extrapolated=round(lp_s * B, 1),
                 speedup=round(lp_s * B / (ms * 1e-3), 1), max_rel_diff_vs_linprog=float(np.max(np.abs(got - ref) / np.abs(ref))),
                 gpu=name, power_limit=power)
        print(json.dumps(r), flush=True)
        results.append(r)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
