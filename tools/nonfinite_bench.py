#!/usr/bin/env python
"""The cost of the non-finite step guard, GNNAETrainer(nonfinite="skip"), on one GPU, and an A/B of the four solver kernels that gained
a non-finite input check.

Step time: CLI-default architecture (config.build_models, seed 0), bf16 mode, CUDA graphs, synthetic_jets inputs in pinned host memory,
Chamfer loss, Adam; at N = 30 / B = 4096 and N = 150 / B = 2048 a trainer with nonfinite="ignore" and one with "skip".  After two warm-up
steps each, --rounds rounds alternate the two; a round times --steps calls of step() (each ends in its host read of the loss) with
CUDA events.  Also timed alone: the two guard launches (gj_nonfinite_flag, gj_nonfinite_check over the n + 1 gradient floats), 200
launches each.

Solver A/B (--before PATH, a libgnnjet_b200.so built from the parent commit): that library and the in-tree one loaded into this
process, the same inputs, rounds alternating the two; per round --solver-calls launches timed with CUDA events.  Kernels: gj_emd and
gj_emd_loss (polar synthetic_jets), gj_assignment and gj_hungarian_mse_loss (absolute Cartesian), each at N = 30 / B = 4096 and
N = 150 / B = 2048.  Every output of both libraries is compared bit for bit.

Median, min and max over the rounds; the card's name and power limit are read in the same run.
GPU box: python tools/nonfinite_bench.py [--before path/to/parent/libgnnjet_b200.so] [--out result.json]"""
import argparse
import ctypes as C
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from gnn_jet_autoencoder_b200 import GNNAETrainer, _lib
from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models
from gnn_jet_autoencoder_b200.trainer import synthetic_jets

SHAPES = ((30, 4096), (150, 2048))


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def summary(v):
    return dict(median=round(statistics.median(v), 4), min=round(min(v), 4), max=round(max(v), 4))


def event_ms(fn, calls):
    """Mean milliseconds per call of ``fn`` over ``calls`` calls, CUDA events around them."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / calls


def bench_steps(args):
    out = {}
    for N, B in SHAPES:
        trainers = {}
        for mode in ("ignore", "skip"):
            enc, dec = build_models(N, DEFAULT_ARCH, device="cuda:0", precision="bf16", seed=0)
            trainers[mode] = GNNAETrainer(enc, dec, batch_size=B, nonfinite=mode)
        xs = [torch.from_numpy(synthetic_jets(B, N, seed=200 + i)).pin_memory() for i in range(4)]
        for tr in trainers.values():
            tr.step(xs[0])
            tr.step(xs[1])
        times = {k: [] for k in trainers}
        for _ in range(args.rounds):
            for k, tr in trainers.items():
                times[k].append(event_ms(lambda: tr.step(xs[2]), args.steps))
        tr = trainers["skip"]
        st = torch.cuda.current_stream().cuda_stream
        lib = tr.lib
        flag = lambda: lib.gj_nonfinite_flag(tr.stats.data_ptr(), 3, tr.grad_buffer.data_ptr() + 4 * tr.grad.numel(), st)
        check = lambda: lib.gj_nonfinite_check(tr.grad_buffer.data_ptr(), tr.grad_buffer.numel(), tr.guard.data_ptr(),
                                               tr.stats.data_ptr() + 24, st)
        med = {k: statistics.median(v) for k, v in times.items()}
        out[f"N{N}_B{B}"] = dict(step_ms={k: summary(v) for k, v in times.items()},
                                 skip_minus_ignore_ms=round(med["skip"] - med["ignore"], 4),
                                 launches_per_step={k: t.launches_per_step for k, t in trainers.items()},
                                 flag_launch_us=round(1e3 * event_ms(flag, 200), 2), check_launch_us=round(1e3 * event_ms(check, 200), 2),
                                 gradient_floats=tr.grad_buffer.numel(), applied_steps=tr.applied_steps, nonfinite_steps=tr.nonfinite_steps)
        del trainers
        torch.cuda.empty_cache()
    return out


def load_copy(path, tag):
    """A private copy of a library file loaded with the signatures of _lib (two copies of one library coexist in a process)."""
    d = tempfile.mkdtemp(prefix="gj_ab_")
    dst = os.path.join(d, f"libgnnjet_b200_{tag}.so")
    shutil.copyfile(path, dst)
    lib = C.CDLL(dst)
    for name in ("gj_emd", "gj_emd_loss", "gj_emd_loss_workspace", "gj_assignment", "gj_hungarian_mse_loss",
                 "gj_hungarian_mse_loss_workspace", "gj_last_error"):
        res, argt = _lib.SIGNATURES[name]
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, argt
    return lib, d


def solver_cases(N, B):
    """name -> (make outputs, launch(lib, outs)) for the four kernels at this shape."""
    dev = "cuda:0"
    st = torch.cuda.current_stream().cuda_stream
    p = torch.from_numpy(synthetic_jets(B, N, seed=300)).to(dev)
    q = torch.from_numpy(synthetic_jets(B, N, seed=301)).to(dev)
    g = torch.Generator().manual_seed(302)
    a = torch.randn((B, N, 3), generator=g).to(dev)
    b = torch.randn((B, N, 3), generator=g).to(dev)
    f64 = dict(device=dev, dtype=torch.float64)

    def chk(rc, lib, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {lib.gj_last_error().decode()}")

    def emd_outs():
        return dict(emd=torch.zeros(B, **f64), dp=torch.zeros((B, N, 3), device=dev), pot=torch.zeros((B, 2 * N + 2), **f64),
                    status=torch.zeros(B, device=dev, dtype=torch.int32))

    def emd_run(lib, o):
        chk(lib.gj_emd(B, N, N, p.data_ptr(), q.data_ptr(), 1.0, 1.0, 0, o["emd"].data_ptr(), None, o["dp"].data_ptr(), o["pot"].data_ptr(),
                       o["status"].data_ptr(), None, 0, st), lib, "gj_emd")

    ws_bytes = max(int(_lib.load().gj_emd_loss_workspace(B, N)), int(_lib.load().gj_hungarian_mse_loss_workspace(B, N)))

    def loss_outs():
        return dict(terms=torch.zeros(3, device=dev), failed=torch.zeros(1, device=dev), dp=torch.zeros((B, N, 3), device=dev),
                    ws=torch.zeros(ws_bytes, dtype=torch.uint8, device=dev), match=torch.zeros((B, N), device=dev, dtype=torch.int32))

    def emd_loss_run(lib, o):
        chk(lib.gj_emd_loss(B, N, 3, _lib.GJ_EMD_COORDS_POLAR, p.data_ptr(), q.data_ptr(), 1.0, 1.0, 0, 1.0, o["terms"].data_ptr(),
                            o["failed"].data_ptr(), o["dp"].data_ptr(), o["ws"].data_ptr(), ws_bytes, st), lib, "gj_emd_loss")

    def asg_outs():
        return dict(match=torch.zeros((B, N), device=dev, dtype=torch.int32), total=torch.zeros(B, device=dev))

    def asg_run(lib, o):
        chk(lib.gj_assignment(B, N, 3, 0, a.data_ptr(), b.data_ptr(), o["match"].data_ptr(), o["total"].data_ptr(), st), lib, "gj_assignment")

    def hmse_run(lib, o):
        chk(lib.gj_hungarian_mse_loss(B, N, 3, _lib.GJ_HMSE_ABS_CARTESIAN, a.data_ptr(), b.data_ptr(), 1.0 / (B * N * 3), o["terms"].data_ptr(),
                                      o["dp"].data_ptr(), o["match"].data_ptr(), o["ws"].data_ptr(), ws_bytes, st), lib, "gj_hungarian_mse_loss")

    return {"gj_emd": (emd_outs, emd_run), "gj_emd_loss": (loss_outs, emd_loss_run), "gj_assignment": (asg_outs, asg_run),
            "gj_hungarian_mse_loss": (loss_outs, hmse_run)}


def bench_solvers(args):
    before, d0 = load_copy(args.before, "before")
    after, d1 = load_copy(_lib.LIB_PATH, "after")
    libs = {"before": before, "after": after}
    out = {}
    try:
        for N, B in SHAPES:
            for kname, (make, run) in solver_cases(N, B).items():
                outs = {k: make() for k in libs}
                for k, lib in libs.items():
                    run(lib, outs[k])
                torch.cuda.synchronize()
                same = all(torch.equal(outs["before"][f], outs["after"][f]) for f in outs["before"])
                calls = args.solver_calls if N == 30 else max(2, args.solver_calls // 10)
                times = {k: [] for k in libs}
                for _ in range(args.rounds):
                    for k, lib in libs.items():
                        times[k].append(event_ms(lambda: run(lib, outs[k]), calls))
                med = {k: statistics.median(v) for k, v in times.items()}
                out[f"{kname}_N{N}_B{B}"] = dict(ms={k: summary(v) for k, v in times.items()}, outputs_bitwise_equal=same,
                                                  change_pct=round(100 * (med["after"] / med["before"] - 1), 2), calls_per_round=calls)
                print(kname, N, B, out[f"{kname}_N{N}_B{B}"], flush=True)
    finally:
        shutil.rmtree(d0, ignore_errors=True)
        shutil.rmtree(d1, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--solver-calls", type=int, default=20)
    ap.add_argument("--before", default=None, help="libgnnjet_b200.so built from the parent commit (solver A/B)")
    ap.add_argument("--skip-steps", action="store_true", help="only the solver A/B")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("nonfinite_bench.py needs a CUDA device")
    name, power = gpu_info()
    out = dict(gpu=name, power_limit=power, rounds=args.rounds)
    if args.before:
        out["solver_ab"] = bench_solvers(args)
    if not args.skip_steps:
        out["steps"] = bench_steps(args)
        out["steps_per_round"] = args.steps
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
