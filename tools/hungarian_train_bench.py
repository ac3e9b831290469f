#!/usr/bin/env python
"""Training with the Hungarian-matched MSE: GNNAETrainer.compute_gradients() with loss_choice="hungarian" against "chamfer" and
"emd", the gj_hungarian_mse_loss launch alone and HungarianMSELoss forward + backward through autograd, on one GPU.

CLI-default architecture (config.build_models, seed 0) in the bf16 mode, polar_coord=True, synthetic_jets inputs ([pt, eta, phi],
zero padded), CUDA graphs on.  The Hungarian loss runs in HungarianMSELoss's default coordinates (absolute, Cartesian: the features
as they are), the EMD as EMDLoss(R=1, beta=1, reduction="sum").  After a warm-up (graph capture), each round times --calls calls of
the Chamfer step, the Hungarian step, the EMD step, the Hungarian launch alone and the unfused HungarianMSELoss (the last two on
the Hungarian trainer's reconstruction and input), with CUDA events; --rounds rounds alternate the five.  Reported: median, min and
max over the rounds of the per-call time.
GPU box: python tools/hungarian_train_bench.py [--out result.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from gnn_jet_autoencoder_b200 import EMDLoss, GNNAETrainer, HungarianMSELoss, _lib
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


def timed(fn, calls):
    """ms per call of ``fn`` over ``calls`` back-to-back calls, CUDA events around the window."""
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(calls):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / calls


def summary(v):
    return dict(median=round(statistics.median(v), 3), min=round(min(v), 3), max=round(max(v), 3))


def run(N, B, calls, rounds, precision):
    dev = torch.device("cuda", 0)
    x = torch.from_numpy(synthetic_jets(B, N, seed=1234)).pin_memory()
    trainers = {}
    for loss in ("chamfer", "hungarian", "emd"):
        enc, dec = build_models(N, DEFAULT_ARCH, device=dev, precision=precision, seed=0)
        kw = dict(emd_loss=EMDLoss(R=1.0, beta=1.0, polar_coord=True, reduction="sum")) if loss == "emd" else {}
        tr = GNNAETrainer(enc, dec, batch_size=B, loss_choice=loss, polar_coord=True, **kw)
        tr.load_batch(x)
        tr.compute_gradients()           # eager warm-up + graph capture
        tr.compute_gradients()
        trainers[loss] = tr
    th = trainers["hungarian"]
    lib, st = _lib.load(), torch.cuda.current_stream().cuda_stream
    terms = torch.empty(3, device=dev)
    dp = torch.empty_like(th.recon)

    def hungarian_launch():
        _lib.check(lib.gj_hungarian_mse_loss(B, N, 3, _lib.GJ_HMSE_ABS_CARTESIAN, th.recon.data_ptr(), th.x.data_ptr(), th.hmse_scale,
                                             terms.data_ptr(), dp.data_ptr(), None, th.ws.data_ptr(), th.ws_bytes, st),
                   "gj_hungarian_mse_loss")

    recon = th.recon.detach().clone()

    def hungarian_autograd():
        r = recon.clone().requires_grad_()
        HungarianMSELoss()(r, th.x).backward()

    hungarian_launch()
    hungarian_autograd()
    torch.cuda.synchronize()
    times = {"chamfer_step": [], "hungarian_step": [], "emd_step": [], "hungarian_launch": [], "hungarian_autograd": []}
    for _ in range(rounds):
        times["chamfer_step"].append(timed(trainers["chamfer"].compute_gradients, calls))
        times["hungarian_step"].append(timed(th.compute_gradients, calls))
        times["emd_step"].append(timed(trainers["emd"].compute_gradients, calls))
        times["hungarian_launch"].append(timed(hungarian_launch, calls))
        times["hungarian_autograd"].append(timed(hungarian_autograd, calls))
    med = {k: statistics.median(v) for k, v in times.items()}
    out = dict(N=N, B=B, precision=precision, calls_per_round=calls, rounds=rounds,
               **{f"{k}_ms": summary(v) for k, v in times.items()},
               hungarian_step_over_chamfer_step=round(med["hungarian_step"] / med["chamfer_step"], 2),
               emd_step_over_chamfer_step=round(med["emd_step"] / med["chamfer_step"], 2),
               hungarian_jets_per_s=round(B / med["hungarian_launch"] * 1e3),
               hungarian_loss=float(th.stats[2].item()), chamfer_loss=float(trainers["chamfer"].stats[2].item()))
    del trainers, th
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("hungarian_train_bench.py needs a CUDA device")
    name, power = gpu_info()
    results = []
    for N, B in ((30, 4096), (150, 2048)):
        r = dict(run(N, B, args.calls, args.rounds, args.precision), gpu=name, power_limit=power)
        print(json.dumps(r), flush=True)
        results.append(r)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
