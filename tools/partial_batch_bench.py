#!/usr/bin/env python
"""The cost of a short last batch in GNNAETrainer(partial_batches=True), on one GPU.

CLI-default architecture (config.build_models, seed 0) in the bf16 mode, N = 30, batch_size = 4096, synthetic_jets inputs in pinned
host memory, CUDA graphs on.  Reported:
- the constructor with and without the flag (with it, the buffers are sized for every batch of up to batch_size jets);
- the one-time cost of the tail: the first step of a 1000-jet batch (plan + eager warm-up + graph capture + replay) against a
  later step of that size, host clock around synchronised steps;
- steady-state training epochs (run_epoch, outputs collected): 40 full batches plus the tail against the same 40 batches without
  it on the same trainer, and the 40 batches on a trainer without the flag; --rounds rounds alternate the three after a warm-up
  epoch of each; median, min and max over the rounds;
- device memory each trainer holds, and the card's name and power limit, read in the same run.
GPU box: python tools/partial_batch_bench.py [--out result.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from gnn_jet_autoencoder_b200 import GNNAETrainer
from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models
from gnn_jet_autoencoder_b200.trainer import synthetic_jets


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def wall_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def summary(v):
    return dict(median=round(statistics.median(v), 3), min=round(min(v), 3), max=round(max(v), 3))


def build(N, B, precision, partial):
    enc, dec = build_models(N, DEFAULT_ARCH, device="cuda:0", precision=precision, seed=0)
    before = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    tr = GNNAETrainer(enc, dec, batch_size=B, partial_batches=partial)
    return tr, (time.perf_counter() - t0) * 1e3, torch.cuda.memory_allocated() - before


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batches", type=int, default=40)
    ap.add_argument("--tail", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("partial_batch_bench.py needs a CUDA device")
    N, B = 30, 4096
    name, power = gpu_info()
    batches = [torch.from_numpy(synthetic_jets(B, N, seed=100 + i)).pin_memory() for i in range(args.batches)]
    tail = torch.from_numpy(synthetic_jets(args.tail, N, seed=99)).pin_memory()

    fixed, ctor_fixed_ms, mem_fixed = build(N, B, args.precision, False)
    tr, ctor_partial_ms, mem_partial = build(N, B, args.precision, True)
    for t in (fixed, tr):
        t.step(batches[0])                 # full-size graph
        t.step(batches[1])
    mem_before_tail = torch.cuda.memory_allocated()
    first_tail_ms = wall_ms(lambda: tr.step(tail))
    later_tail_ms = [wall_ms(lambda: tr.step(tail)) for _ in range(5)]
    full_step_ms = [wall_ms(lambda: tr.step(batches[2])) for _ in range(5)]
    tail_adds_bytes = torch.cuda.memory_allocated() - mem_before_tail

    epochs = {"with_tail": lambda: tr.run_epoch(batches + [tail]), "without_tail": lambda: tr.run_epoch(batches),
              "without_flag": lambda: fixed.run_epoch(batches)}
    for fn in epochs.values():                 # pinned epoch buffers
        fn()
    times = {k: [] for k in epochs}
    for _ in range(args.rounds):
        for k, fn in epochs.items():
            times[k].append(wall_ms(fn))
    med = {k: statistics.median(v) for k, v in times.items()}
    out = dict(gpu=name, power_limit=power, N=N, batch_size=B, tail=args.tail, batches=args.batches, precision=args.precision,
               rounds=args.rounds, constructor_ms=dict(without_flag=round(ctor_fixed_ms, 1), with_flag=round(ctor_partial_ms, 1)),
               trainer_device_bytes=dict(without_flag=mem_fixed, with_flag=mem_partial),
               tail_plan_adds_device_bytes=tail_adds_bytes,
               first_tail_step_ms=round(first_tail_ms, 2), later_tail_step_ms=summary(later_tail_ms),
               one_time_tail_cost_ms=round(first_tail_ms - statistics.median(later_tail_ms), 2), full_step_ms=summary(full_step_ms),
               **{f"epoch_{k}_ms": summary(v) for k, v in times.items()},
               tail_adds_ms=round(med["with_tail"] - med["without_tail"], 3),
               flag_costs_on_full_batches_ms=round(med["without_tail"] - med["without_flag"], 3),
               jets_per_s=dict(with_tail=round((args.batches * B + args.tail) / med["with_tail"] * 1e3),
                               without_tail=round(args.batches * B / med["without_tail"] * 1e3)))
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
