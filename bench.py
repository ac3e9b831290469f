#!/usr/bin/env python
"""Benchmark of the GNNAE train step (BASELINE.json: jets/sec, fwd+bwd+Adam, Chamfer loss, N=30).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--num-nodes 30|150]
                    [--batch B] [--precision bf16|fp32] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  Headline workload: reference CLI-default architecture, synthetic JetNet-shaped
jets, 4096 jets per GPU (BASELINE config 2 at N=1; 8 GPUs = config 4's 32768-jet global batch), weak scaling.
The same line carries a "configs" object with the other BASELINE configurations measured in the same run: config 3
(N=150, B=2048), config 2 in the fp32 parity mode, the CPU forward of config 1 and the CPU N=150 train step, the
reference op sequence (oracle/torch_port.py) on the same GPU, config 4 as specified (global batch 32768: one GPU as the
denominator at --gpus 1, sharded B/G per rank at --gpus G, "strong") and a few points of config 5's deep / wide sweep;
at --gpus G > 1 also "dp_parity" (parameters bit-identical across ranks, G-rank gradient = one-rank gradient).
"value" times the step with the batch resident in HBM (CUDA events, L2 flushed between steps, max over
ranks); "e2e" goes through the public ``GNNAETrainer.step`` with a pinned host batch per step and a
device->host read of the loss.  ``--impl reference`` times the CPU PyTorch restatement of the reference's
train step (oracle/torch_port.py, "port") on the host cores.
``--dump-outputs DIR`` also writes what the last timed step computed as DIR/<name>.npy (``dump_timed_outputs``); inputs and
initial parameters are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "jets/sec fwd+bwd GNNAE train step"
UNIT = "jets/s"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(burst=float(p["bf16_tflops"]), sustained=float(p["bf16_tflops_sustained"]), hbm=float(p["hbm_gbs"]),
                    source="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------------------------------
# CPU baseline: torch-CPU restatement of the reference step on a bounded sample
# --------------------------------------------------------------------------------------------------
def cpu_reference_step_rate(num_nodes, sample_jets, steps, warmup, budget_s=25.0):
    import torch
    from gnn_jet_autoencoder_b200.trainer import synthetic_jets
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, *_ = _port_step(num_nodes, torch.device("cpu"))
    x = torch.from_numpy(synthetic_jets(sample_jets, num_nodes, seed=1234))
    for _ in range(max(1, warmup)):
        step.step(x)
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        step.step(x)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return dict(value=done * sample_jets / dt, unit=UNIT, cores=cores, kind="port",
                sample=f"{done} steps of {sample_jets} jets (N={num_nodes}) through oracle/torch_port.py "
                       f"(torch {torch.__version__} CPU, fp32, autograd + 2x Adam), {dt:.1f} s"), dt / done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.cpu_sample or (256 if args.num_nodes <= 32 else 16)
    cb, sec_per_step = cpu_reference_step_rate(args.num_nodes, sample, args.steps, min(args.warmup, 2), budget_s=120.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args, sample, 1),
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, per_gpu_batch, world):
    return {"workload": f"GNNAE full training step (fwd+bwd+Adam, Chamfer loss) N={args.num_nodes} "
                        f"batch {per_gpu_batch} per GPU (BASELINE config {'2' if args.num_nodes == 30 else '3'})",
            "arch": "reference CLI defaults: edge [32,128,64,16], node [[16],[32],[8]], 3 MP steps, latent 20 'mean'",
            "num_nodes": args.num_nodes, "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * world,
            "parallelism": f"dp{world} (batch shard, one flat-gradient all-reduce)",
            "l2": "flushed between timed steps (256 MiB write, outside the timed events)"}


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            parts = [c.strip() for c in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}



# --------------------------------------------------------------------------------------------------
# the other BASELINE configurations, measured in the same run ("configs" of the JSON line)
# --------------------------------------------------------------------------------------------------
def _time_trainer(tr, host, steps, warmup, flush, barrier=None, rank_max=None):
    """ms per step with the batch resident in HBM (CUDA events per step, L2 flushed in between)."""
    import torch
    tr.load_batch(host)
    for _ in range(max(warmup, 3)):
        tr.compute_gradients()
        tr.apply_gradients()
    (barrier or torch.cuda.synchronize)()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s, e in ev:
        flush.fill_(1)
        s.record()
        tr.compute_gradients()
        tr.apply_gradients()
        e.record()
    (barrier or torch.cuda.synchronize)()
    ms = sum(s.elapsed_time(e) for s, e in ev)
    return (rank_max(ms) if rank_max else ms) / steps


def _train_config(N, B, precision, dev, flush, steps, arch=None, group=None, world=1, barrier=None, rank_max=None, seed=1234):
    import torch
    from gnn_jet_autoencoder_b200 import GNNAETrainer, synthetic_jets
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models, train_flops_per_jet
    arch = arch or DEFAULT_ARCH
    # build + warm-up (kernel loading, CUDA-graph capture) carry no collective; the ranks then agree that every one of them got
    # through before the first barrier, so that a failure on one rank is reported instead of leaving the others in a collective
    err, tr, host = None, None, None
    try:
        enc, dec = build_models(N, arch, device=dev, precision=precision, seed=0)
        tr = GNNAETrainer(enc, dec, batch_size=B, process_group=group)
        host = torch.from_numpy(synthetic_jets(B, N, seed=seed)).pin_memory()
        tr.load_batch(host)
        tr.compute_gradients()
        torch.cuda.synchronize()
    except Exception as ex:
        err = ex
    if world > 1:
        import torch.distributed as dist
        ok = torch.tensor([0.0 if err is not None else 1.0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() < 1.0 and err is None:
            err = RuntimeError("another rank failed while building / capturing this configuration")
    if err is not None:
        del tr
        torch.cuda.empty_cache()
        raise err
    ms = _time_trainer(tr, host, steps, 3, flush, barrier, rank_max)
    value = world * B / (ms * 1e-3)
    peaks = measured_peaks()
    tf = value / world * train_flops_per_jet(N, arch) / 1e12
    out = {"value": value, "unit": UNIT, "ms_per_step": ms, "num_nodes": N, "per_gpu_batch": B, "global_batch": B * world,
           "dtype": "bf16" if precision == "bf16" else "fp32",
           "step_roofline_frac": tf / peaks["sustained"], "tflops_per_gpu": tf}
    del tr, enc, dec
    torch.cuda.empty_cache()
    return out


def _cpu_forward_config1(budget_s=8.0):
    """BASELINE config 1: encoder + decoder forward, N=30, B=256, fp32, no_grad, on the host cores (reference op sequence)."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch_port as TP
    step, enc_cfg, dec_cfg, ep, dp = _port_step(30, torch.device("cpu"))
    x = torch.from_numpy(__import__("gnn_jet_autoencoder_b200").synthetic_jets(256, 30, seed=1234))
    with torch.no_grad():
        for _ in range(2):
            TP.decoder_forward(TP.encoder_forward(x, step.enc_p, enc_cfg), step.dec_p, dec_cfg)
        t0, n = time.perf_counter(), 0
        while n < 5 or (time.perf_counter() - t0 < budget_s and n < 20):
            TP.decoder_forward(TP.encoder_forward(x, step.enc_p, enc_cfg), step.dec_p, dec_cfg)
            n += 1
        dt = time.perf_counter() - t0
    return {"value": n * 256 / dt, "unit": "jets/s (forward only)", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"{n} forwards of 256 jets (N=30), oracle/torch_port.py, torch CPU fp32, {dt:.1f} s"}


def _port_step(num_nodes, device):
    """The reference's train step restated with stock torch ops (oracle/torch_port.py) with the CLI-default architecture."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch_port as TP
    from golden_cases import _linear
    import gnnae_oracle as O
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH as A
    rng = np.random.default_rng(0)
    enc_cfg = dict(num_nodes=num_nodes, input_node_size=A["vec_dims"], latent_node_size=A["latent_node_size"],
                   node_sizes=A["node_sizes"], edge_sizes=A["edge_sizes"], num_mps=A["num_mps"], alphas=A["alphas"],
                   latent_map=A["latent_map"])
    dec_cfg = dict(enc_cfg, output_node_size=A["vec_dims"])
    ep = O.init_graphnet_params(rng, A["vec_dims"], A["latent_node_size"], A["node_sizes"], A["edge_sizes"], A["num_mps"],
                                prefix="encoder.", dtype=np.float32)
    h0 = A["node_sizes"][0][0]
    dp = {}
    dp["linear.weight"], dp["linear.bias"] = _linear(rng, num_nodes * h0, A["latent_node_size"])
    dp.update(O.init_graphnet_params(rng, h0, A["vec_dims"], A["node_sizes"], A["edge_sizes"], A["num_mps"],
                                     prefix="decoder.", dtype=np.float32))
    mk = lambda d: {k: torch.tensor(v, dtype=torch.float32, device=device, requires_grad=True) for k, v in d.items()}
    return TP.TorchTrainStep(mk(ep), mk(dp), enc_cfg, dec_cfg), enc_cfg, dec_cfg, ep, dp


def _gpu_reference(dev, num_nodes=30):
    """The reference's op sequence (materialised (B,N,N,2H+1) tensor, autograd, two Adams) with stock torch CUDA ops on the same
    GPU, fp32, at the largest power-of-two batch <= 4096 that fits (11.3 MB of saved activations per jet at N=30)."""
    import torch
    from gnn_jet_autoencoder_b200 import synthetic_jets
    B = 4096 if num_nodes <= 32 else 64
    while B >= 16:
        try:
            step, *_ = _port_step(num_nodes, dev)
            x = torch.from_numpy(synthetic_jets(B, num_nodes, seed=1234)).to(dev)
            for _ in range(2):
                step.step(x)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = 5
            for _ in range(n):
                step.step(x)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / n
            del step, x
            torch.cuda.empty_cache()
            return {"value": B / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "batch": B, "num_nodes": num_nodes, "dtype": "fp32",
                    "what": "oracle/torch_port.py: the reference's op sequence on stock torch CUDA kernels (cuBLAS SIMT fp32 + elementwise), "
                            "same B200, wall clock around step() incl. its loss.item() sync"}
        except torch.cuda.OutOfMemoryError:
            torch.cuda.empty_cache()
            B //= 2
    return {"unavailable": "out of memory at every batch size tried"}


def _sweep_points(dev, flush, world, group, barrier, rank_max, N=30, B=2048):
    """A few members of BASELINE config 5 (num_mps 3-6, hidden 64-256 with node_sizes [[H]] / edge_sizes [[H, H]], latent 1-64)."""
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH
    out = []
    for num_mps, H, latent in [(3, 64, 8), (6, 64, 1), (3, 128, 8), (4, 128, 64), (3, 256, 16)]:
        arch = dict(DEFAULT_ARCH, edge_sizes=[[H, H]], node_sizes=[[H]], num_mps=num_mps, latent_node_size=latent)
        try:
            r = _train_config(N, B if H < 256 else B // 4, "bf16", dev, flush, 4, arch=arch, group=group, world=world, barrier=barrier,
                              rank_max=rank_max)
            out.append(dict(num_mps=num_mps, hidden=H, latent=latent, **{k: r[k] for k in ("value", "ms_per_step", "per_gpu_batch",
                                                                                           "step_roofline_frac")}))
        except Exception as ex:      # widths the kernels do not cover are reported, not hidden
            out.append(dict(num_mps=num_mps, hidden=H, latent=latent, error=f"{type(ex).__name__}: {str(ex)[:120]}"))
    return out


def _dp_parity(dev, world, rank, precision):
    """G-rank data parallelism against one rank on the concatenated batch: the all-reduced flat gradient of a small sharded batch,
    and (by the caller) bit-identical parameters after the timed steps."""
    import torch
    import torch.distributed as dist
    from gnn_jet_autoencoder_b200 import GNNAETrainer, synthetic_jets
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models
    from gnn_jet_autoencoder_b200.trainer import allreduce_flat_, shard_range
    per, N = 8, 30
    xg = torch.from_numpy(synthetic_jets(per * world, N, seed=77))
    lo, hi = shard_range(per * world, rank, world)
    enc, dec = build_models(N, DEFAULT_ARCH, device=dev, precision=precision, seed=0)
    tr = GNNAETrainer(enc, dec, batch_size=hi - lo, use_cuda_graph=False)
    tr.load_batch(xg[lo:hi])
    tr.compute_gradients()
    allreduce_flat_(tr.grad)
    g_dp = tr.grad.clone()
    err = None
    if rank == 0:
        enc1, dec1 = build_models(N, DEFAULT_ARCH, device=dev, precision=precision, seed=0)
        tr1 = GNNAETrainer(enc1, dec1, batch_size=per * world, use_cuda_graph=False)
        tr1.load_batch(xg)
        tr1.compute_gradients()
        torch.cuda.synchronize()
        err = float((g_dp - tr1.grad).norm() / tr1.grad.norm())
    dist.barrier()
    return err


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_timed_outputs(tr, out_dir, limit=DUMP_LIMIT_BYTES):
    """Write what the last timed step (compute_gradients + apply_gradients) hands a caller to ``out_dir``/<name>.npy:
    latent (B, latent) and recon (B, N, F) of its forward pass, loss (float64, the value ``GNNAETrainer.step`` returns), grad
    (the flat parameter gradient) and params (the flat parameters after the optimiser update), all float32 but the loss.
    Above ``limit`` bytes in all, latent and recon keep a fixed sample of jets: the sorted rows
    ``numpy.random.default_rng(0).choice(B, k, replace=False)``, the same for every build at the same arguments."""
    import numpy as np
    out = {"latent": tr.latent, "recon": tr.recon, "grad": tr.grad, "params": tr.flat}
    out = {k: v.detach().cpu().numpy().astype(np.float32, copy=False) for k, v in out.items()}
    out["loss"] = np.float64(tr.loss_from_stats(tr.stats.cpu()))
    per_jet = out["latent"][0].nbytes + out["recon"][0].nbytes
    fixed = out["grad"].nbytes + out["params"].nbytes + 8 + 128 * len(out)      # + the .npy headers
    k = min(tr.B, (limit - fixed) // per_jet)
    if k < tr.B:
        rows = np.sort(np.random.default_rng(0).choice(tr.B, k, replace=False))
        out["latent"], out["recon"] = out["latent"][rows], out["recon"][rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)

# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from gnn_jet_autoencoder_b200 import GNNAETrainer, ops, synthetic_jets
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models, edge_macs_per_row, train_flops_per_jet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the path has no CPU fallback")
    # Last-resort guard for multi-rank runs: a rank stuck in a collective (a peer died, NCCL teardown hangs) would keep the whole job
    # alive until the launcher's limit.  At the deadline rank 0 prints the line it has (the headline measurement comes first, the extra
    # "configs" last) and every rank leaves.
    state = {"line": None, "printed": False}
    def _deadline():
        if rank == 0 and state["line"] is not None and not state["printed"]:
            state["line"]["configs_incomplete"] = "deadline reached while measuring the extra configurations"
            print(json.dumps(state["line"]), flush=True)
        os._exit(0 if (rank != 0 or state["line"] is not None) else 1)
    if world > 1:
        import threading
        guard = threading.Timer(float(os.environ.get("GNNJET_BENCH_DEADLINE_S", "420")), _deadline)
        guard.daemon = True
        guard.start()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries ONE JSON line: NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION) is dropped, any more verbose
        # debug level the caller asked for goes to stderr
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    N = args.num_nodes
    B = args.batch or (4096 if N <= 32 else 2048)
    enc, dec = build_models(N, DEFAULT_ARCH, device=dev, precision=args.precision, seed=0)
    tr = GNNAETrainer(enc, dec, batch_size=B, use_cuda_graph=not args.no_graph)
    # a few distinct pinned host batches (seed = 1234 + rank, SURVEY.md 8.d), cycled by the e2e loop
    host = [torch.from_numpy(synthetic_jets(B, N, seed=1234 + rank + 101 * i)).pin_memory() for i in range(4)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(v):
        if world > 1:
            t = torch.tensor([v], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    # ---- warm-up (also builds the CUDA graph) ----
    tr.load_batch(host[0])
    for _ in range(max(args.warmup, 3)):
        tr.compute_gradients()
        tr.apply_gradients()
    barrier()

    # ---- device-resident timing: K steps, events around each step, L2 flushed in between ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = ops.LAUNCHES["count"]
    barrier()
    for s, e in ev:
        flush.fill_(1)
        s.record()
        tr.compute_gradients()
        tr.apply_gradients()
        e.record()
    barrier()
    if args.dump_outputs and rank == 0:      # before the e2e loop below moves the parameters on
        dump_timed_outputs(tr, args.dump_outputs)
    launches = ops.LAUNCHES["count"] - launches0
    ms_total = rank_max(sum(s.elapsed_time(e) for s, e in ev))
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)

    # ---- end to end: pinned host batch in, loss out, every step, through the public API ----
    for i in range(2):
        tr.step(host[i % len(host)])
    barrier()
    s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    last = 0.0
    for i in range(args.steps):
        last = tr.step(host[i % len(host)])
    e0.record()
    barrier()
    e2e_ms = rank_max(s0.elapsed_time(e0)) / args.steps
    clocks = sampler.stop() if rank == 0 else None

    # ---- dominant kernel alone: backward of the heaviest step (encoder step 1), CUDA events on its stream ----
    peaks = measured_peaks()
    kern = time_dominant_kernel(tr, args) if rank == 0 else None
    if world > 1:
        dist.barrier()

    # ---- the headline line (rank 0); the extra configurations are filled in below as they complete ----
    d2h_bytes = tr.stats_host.numel() * 4
    configs = {}
    if rank == 0:
        flops_jet = train_flops_per_jet(N, DEFAULT_ARCH)
        step_tflops = value / world * flops_jet / 1e12          # per GPU
        state["line"] = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "fp32", "data": "synthetic",
            "config": workload_config(args, B, world),
            "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": B * N * 3 * 4, "d2h_bytes_per_step": d2h_bytes,
                    "api": "GNNAETrainer.step(pinned host batch) -> float loss"},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": kern and {
                "bound": "tensor", "achieved": kern["tflops"], "peak": peaks["burst"], "unit": "TFLOP/s",
                "frac": kern["tflops"] / peaks["burst"], "traffic": kernel_traffic(args, B, N), "kernel": kern["name"],
                "us_per_launch": kern["us"], "algorithmic_flop_per_launch": kern["flop"], "peak_source": peaks["source"] + ", burst",
            },
            "step_roofline": {"bound": "tensor", "achieved": step_tflops, "peak": peaks["sustained"], "unit": "TFLOP/s",
                              "frac": step_tflops / peaks["sustained"], "flop_per_jet": flops_jet,
                              "peak_source": peaks["source"] + ", sustained", "note": "whole train step, per GPU, edge-MLP "
                              "dense-formulation FLOPs (3 x forward); padding and recomputation not counted"},
            "last_loss": last,
            "configs": configs,
        }

    # ---- the other BASELINE configurations ("configs") and the data-parallel parity check ----
    if world > 1:
        # parameters after the timed steps: bit-identical on every rank (same all-reduced gradient, same fused Adam)
        ref = tr.flat.clone()
        dist.broadcast(ref, 0)
        same = torch.tensor([1.0 if torch.equal(ref, tr.flat) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        err = _dp_parity(dev, world, rank, args.precision)
        if rank == 0:
            state["line"]["dp_parity"] = {"params_bit_identical_across_ranks": bool(same.item() == 1.0), "grad_rel_err_vs_one_rank": err,
                                          "what": f"8 jets per rank, N=30: all-reduced {world}-rank flat gradient vs one rank on the concatenated batch"}
    if not args.no_configs and N == 30 and not args.batch:
        del tr
        torch.cuda.empty_cache()
        if world > 1:      # config 4 as specified: fixed global batch 32768, B/G jets per rank (strong scaling)
            try:
                r = _train_config(30, 32768 // world, args.precision, dev, flush, max(4, args.steps // 2), world=world, barrier=barrier,
                                  rank_max=rank_max, seed=1234 + rank)
                r["scaling"] = "strong"
            except Exception as ex:
                r = {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}
            configs["config4_global32768"] = r
        sweep_worlds = [int(w) for w in os.environ.get("GNNJET_BENCH_SWEEP_WORLDS", "1,8").split(",") if w]
        if world in sweep_worlds:
            configs["config5_sweep"] = {"points": _sweep_points(dev, flush, world, None, barrier, rank_max),
                                        "note": "node_sizes [[H]], edge_sizes [[H, H]], N=30, 2048 jets per GPU (512 at H=256), bf16 mode; "
                                                "roofline fraction on the dense-formulation FLOPs"}
        if world == 1:
            configs["config3_n150_b2048"] = _train_config(150, 2048, "bf16", dev, flush, 6)
            configs["config2_fp32_mode"] = _train_config(30, 4096, "fp32", dev, flush, 4)
            configs["config4_global32768"] = dict(_train_config(30, 32768, args.precision, dev, flush, 4), scaling="strong",
                                                  note="one GPU: the denominator of config 4's 2/4/8-GPU strong scaling")
            configs["gpu_reference"] = _gpu_reference(dev)
            if not args.no_cpu_baseline:
                configs["config1_cpu_forward"] = _cpu_forward_config1()
                cb150, _ = cpu_reference_step_rate(150, 16, steps=3, warmup=1, budget_s=15.0)
                configs["cpu_train_n150_b16"] = cb150

    if rank == 0:
        line = state["line"]
        if world == 1 and not args.no_cpu_baseline:
            sample = args.cpu_sample or (256 if N <= 32 else 16)
            line["cpu_baseline"], _ = cpu_reference_step_rate(N, sample, steps=8, warmup=1, budget_s=20.0)
        print(json.dumps(line), flush=True)
        state["printed"] = True
    if world > 1:
        # NCCL teardown has been seen to hang when a peer is gone: the line is out, leave after a bounded wait
        import threading
        bye = threading.Timer(20.0, lambda: os._exit(0))
        bye.daemon = True
        bye.start()
        try:
            torch.cuda.synchronize()
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass
        sys.stdout.flush()
        os._exit(0)


def kernel_traffic(args, B, N):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, read from the committed summary of
    the `ncu --set full` capture (profiles/kernel_traffic.json, written by tools/ncu_summary.py from the .ncu-rep) -- only if
    that capture was taken at the shape and precision of THIS run; null otherwise."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as f:
            t = json.load(f)["edge_bwd2_kernel"]
        if t["B"] == B and t["N"] == N and t["precision"] == args.precision:
            return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"])
    except Exception:
        pass
    return None


def time_dominant_kernel(tr, args, reps=20):
    import torch
    from gnn_jet_autoencoder_b200 import ops
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH
    # heaviest step: the one with the most edge MACs per row
    steps = tr.enc_steps + tr.dec_steps
    def macs(s):
        d = s["desc"]
        w = [2 * d.node_in + 1] + [d.edge_widths[i] for i in range(d.n_edge_layers)]
        return sum(a * b for a, b in zip(w[:-1], w[1:]))
    idx = max(range(len(tr.enc_steps)), key=lambda i: macs(tr.enc_steps[i]))
    s = tr.enc_steps[idx]
    hin = tr.x if idx == 0 else tr.enc_steps[idx - 1]["out"]
    g = tr.d_enc_out if idx == len(tr.enc_steps) - 1 else tr.enc_steps[idx + 1]["din"]
    din = tr.dx if idx == 0 else s["din"]
    st = torch.cuda.current_stream().cuda_stream
    P, G = tr.flat.data_ptr(), tr.grad.data_ptr()
    saved = s.get("saved")
    saved_ptr = saved.data_ptr() if saved is not None else None
    def launch():
        ops.raw_mp_bwd(s["desc"], hin.data_ptr(), s["e"].data_ptr(), P + 4 * s["off"], g.data_ptr(), din.data_ptr(),
                       G + 4 * s["off"], tr.ws.data_ptr(), tr.ws_bytes, st, saved_ptr)
    from gnn_jet_autoencoder_b200 import _lib
    lib = _lib.load()
    def launch_kernel_only():
        # the fused backward edge kernel ALONE, as the training step runs it (saved forward by-products), on the workspace
        # the full call above has populated
        if saved_ptr:
            return lib.gj_bench_edge_bwd_saved_only(s["desc"], hin.data_ptr(), P + 4 * s["off"], din.data_ptr(), G + 4 * s["off"],
                                                    saved_ptr, tr.ws.data_ptr(), tr.ws_bytes, st)
        return lib.gj_bench_edge_bwd_only(s["desc"], hin.data_ptr(), P + 4 * s["off"], din.data_ptr(), G + 4 * s["off"],
                                          tr.ws.data_ptr(), tr.ws_bytes, st)
    for _ in range(3):
        launch()
    kernel_only = launch_kernel_only() == 0
    fn = launch_kernel_only if kernel_only else launch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    us = a.elapsed_time(b) * 1e3 / reps
    flop = 2.0 * 2.0 * macs(s) * tr.N * tr.N * tr.B       # dgrad + wgrad of the dense formulation
    name = (f"edge_bwd2_kernel (fused recompute + dgrad + wgrad of encoder step {idx}, B={tr.B}, N={tr.N}; launched alone "
            f"through gj_bench_edge_bwd{'_saved' if saved_ptr else ''}_only)") if kernel_only else \
           f"gj_mp_step_bwd (encoder step {idx}, B={tr.B}, N={tr.N}, all of its launches)"
    return dict(name=name, us=us, flop=flop, tflops=flop / (us * 1e-6) / 1e12)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--num-nodes", type=int, default=30)
    ap.add_argument("--batch", type=int, default=0, help="jets per GPU (default 4096 at N=30, 2048 at N=150)")
    ap.add_argument("--precision", default=os.environ.get("GNNJET_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra BASELINE configurations of the 'configs' object")
    ap.add_argument("--cpu-sample", type=int, default=0, help="jets per CPU-baseline step")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
