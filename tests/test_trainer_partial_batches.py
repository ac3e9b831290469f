"""Batches of fewer than ``batch_size`` jets in the fused trainer (``GNNAETrainer(partial_batches=True)``): the host-side shape checks
(CPU), and on the GPU a partial step against a fresh trainer of that size (bitwise, every loss, two latent maps, graph and eager),
the full-size step after it, the epoch loop with a short last batch, the default's fixed shape, memory, bf16 and launch counts."""
import types

import numpy as np
import pytest
import torch

from golden_cases import CASES, make_input, make_params
from gnn_jet_autoencoder_b200 import EMDLoss, ops
from gnn_jet_autoencoder_b200.trainer import GNNAETrainer, synthetic_jets

DEV = "cuda"

# the 'mean' latent on the CLI-default architecture, and the 'local_mix' latent with a larger batch than its golden case
PB_CASES = {"default_b257": CASES["default_b257"], "local_mix_b37": dict(CASES["local_mix_us_n8"], B=37),
            "default_n150_b40": dict(CASES["default_n150"], B=40)}

LOSSES = {
    "chamfer": lambda: dict(loss_choice="chamfer"),
    "mse": lambda: dict(loss_choice="mse"),
    "emd_sum": lambda: dict(loss_choice="emd", emd_loss=EMDLoss(polar_coord=False, reduction="sum")),
    "emd_mean": lambda: dict(loss_choice="emd", emd_loss=EMDLoss(polar_coord=False, reduction="mean")),
    "hungarian_abs_cartesian": lambda: dict(loss_choice="hungarian"),
    "hungarian_rel_polar": lambda: dict(loss_choice="hungarian", hungarian_abs_coord=False, hungarian_polar_coord=True),
}


def rel(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def make_trainer(name, batch_size, precision="fp32", graph=True, loss="chamfer", partial=False):
    """A trainer of golden case ``name`` (its seeded parameters) for ``batch_size`` jets."""
    from gnn_jet_autoencoder_b200 import Decoder, Encoder
    case = PB_CASES[name]
    ep, dp = make_params(case)
    enc = Encoder(**case["enc"], device=DEV, precision=precision)
    dec = Decoder(**case["dec"], device=DEV, precision=precision)
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in ep.items()})
    dec.load_state_dict({k: torch.from_numpy(v) for k, v in dp.items()})
    return GNNAETrainer(enc, dec, batch_size=batch_size, lr=1e-3, encoder_metric=case["metric"], decoder_metric=case["metric"],
                        use_cuda_graph=graph, partial_batches=partial, **LOSSES[loss]())


def copy_state(src, dst):
    """Parameters and optimiser state of ``src`` -> ``dst``."""
    for a in ("flat", "exp_avg", "exp_avg_sq"):
        getattr(dst, a).copy_(getattr(src, a))
    dst.step_count = src.step_count


def batch(name, jets, seed):
    case = PB_CASES[name]
    return torch.from_numpy(synthetic_jets(jets, case["N"], seed=seed)).pin_memory()


def assert_same_step(a, b, loss_a, loss_b):
    torch.cuda.synchronize()
    assert loss_a == loss_b
    assert torch.equal(a.grad, b.grad)
    assert torch.equal(a.stats, b.stats)
    assert torch.equal(a.flat, b.flat)
    assert torch.equal(a.recon, b.recon) and torch.equal(a.latent, b.latent)


def check_partial_then_full(name, Bp, precision="fp32", graph=True, loss="chamfer"):
    """Full step, B'-jet step, full step on a partial-batch trainer, each against a fresh trainer of that size in the same state."""
    B = PB_CASES[name]["B"]
    tr = make_trainer(name, B, precision, graph, loss, partial=True)
    tr.step(torch.from_numpy(make_input(PB_CASES[name])).float().pin_memory())      # the full-size graph exists before the tail's
    tr_p = make_trainer(name, Bp, precision, graph, loss)
    copy_state(tr, tr_p)
    xs = batch(name, Bp, seed=71)
    assert_same_step(tr, tr_p, tr.step(xs), tr_p.step(xs))
    assert tr.recon.shape[0] == Bp and tr.launches_per_step == tr_p.launches_per_step
    tr_f = make_trainer(name, B, precision, graph, loss)
    copy_state(tr, tr_f)
    xf = batch(name, B, seed=72)
    assert_same_step(tr, tr_f, tr.step(xf), tr_f.step(xf))
    assert tr.launches_per_step == tr_f.launches_per_step


# ---------------------------------------------------------------- CPU

def test_batch_shape_checks_on_the_host():
    holder = types.SimpleNamespace(partial_batches=True, batch_size=8, N=5, F=3, world=1)
    jets = lambda *shape: GNNAETrainer._jets_in(holder, torch.zeros(shape))
    assert jets(8, 5, 3) == 8 and jets(40, 3) == 8      # the full size, in any layout, as without the flag
    assert jets(1, 5, 3) == 1 and jets(7, 5, 3) == 7
    for shape in ((0, 5, 3), (9, 5, 3), (4, 6, 3), (4, 5, 4), (20, 3)):
        with pytest.raises(ValueError, match="batch of"):
            jets(*shape)
    holder.world = 2
    with pytest.raises(NotImplementedError, match="data-parallel"):
        jets(7, 5, 3)
    assert jets(8, 5, 3) == 8
    fixed = types.SimpleNamespace(partial_batches=False, batch_size=8, N=5, F=3, world=1)
    assert GNNAETrainer._jets_in(fixed, torch.zeros(7, 5, 3)) == 8      # the copy into the (8, 5, 3) buffer then raises


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("frac", ["one", "odd", "last_but_one"])
@pytest.mark.parametrize("name", ["default_b257", "local_mix_b37"])
@pytest.mark.parametrize("loss", sorted(LOSSES))
def test_partial_step_equals_a_trainer_of_that_size(loss, name, frac, graph):
    B = PB_CASES[name]["B"]
    Bp = {"one": 1, "odd": B // 2 | 1, "last_but_one": B - 1}[frac]
    check_partial_then_full(name, Bp, graph=graph, loss=loss)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_partial_step_at_150_particles(precision):
    """N = 150 runs several j blocks per jet; B' = 23 leaves partial (jet, particle) tiles."""
    prev = ops.set_deterministic(True)
    try:
        check_partial_then_full("default_n150_b40", 23, precision)
    finally:
        ops.set_deterministic(prev)


@pytest.mark.gpu
def test_partial_bf16_step_is_deterministic_and_close_to_fp32():
    name, Bp = "default_b257", 129
    xs = batch(name, Bp, seed=73)
    losses = {}
    for precision in ("fp32", "bf16"):
        tr = make_trainer(name, 257, precision, partial=True)
        losses[precision] = tr.step(xs)
    assert abs(losses["bf16"] - losses["fp32"]) <= 2e-2 * abs(losses["fp32"])
    prev = ops.set_deterministic(True)
    try:
        check_partial_then_full(name, Bp, "bf16")
    finally:
        ops.set_deterministic(prev)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_run_epoch_with_a_short_last_batch(graph):
    name, B, Bp = "default_b257", 257, 100
    batches = [batch(name, B, seed=80), batch(name, B, seed=81), batch(name, Bp, seed=82)]
    tr_a = make_trainer(name, B, graph=graph, partial=True)
    tr_b = make_trainer(name, B, graph=graph, partial=True)
    losses, rec, lat = [], [], []
    for x in batches:
        losses.append(tr_a.step(x))
        rec.append(tr_a.recon.cpu().clone())
        lat.append(tr_a.latent.cpu().clone())
    avg, recons, targets, latents = tr_b.run_epoch(batches, is_train=True)
    assert abs(avg - sum(losses) / 3) <= 1e-6 * abs(avg)
    assert recons.shape[0] == latents.shape[0] == targets.shape[0] == 2 * B + Bp
    assert torch.equal(recons, torch.cat(rec)) and torch.equal(latents, torch.cat(lat))
    assert torch.equal(targets, torch.cat(batches))
    assert torch.equal(tr_a.flat, tr_b.flat)
    # validation: forward + loss only, against forward_only batch by batch
    before = tr_b.flat.clone()
    vavg, vrec, vtgt, vlat = tr_b.run_epoch([b.to(DEV) for b in batches], is_train=False)
    assert torch.equal(tr_b.flat, before)
    vals, rec, lat = [], [], []
    for x in batches:
        z, y = tr_a.forward_only(x)
        tr_a._loss(torch.cuda.current_stream().cuda_stream)
        vals.append(tr_a.loss_from_stats(tr_a.stats.cpu()))
        rec.append(y.cpu())
        lat.append(z.cpu())
    assert abs(vavg - sum(vals) / 3) <= 1e-6 * abs(vavg)
    assert torch.equal(vrec, torch.cat(rec)) and torch.equal(vlat, torch.cat(lat)) and torch.equal(vtgt, torch.cat(batches))
    # a short batch that is not the last one
    with pytest.raises(ValueError, match="only the last batch"):
        tr_b.run_epoch([batches[2], batches[0]])


@pytest.mark.gpu
def test_fixed_shape_by_default_and_bad_batches():
    name, B = "local_mix_b37", 37
    tr = make_trainer(name, B)
    with pytest.raises(RuntimeError):
        tr.step(batch(name, B - 1, seed=90))
    with pytest.raises(ValueError, match="drop the last"):
        tr.run_epoch([batch(name, B - 1, seed=90)])
    tr = make_trainer(name, B, partial=True)
    N = PB_CASES[name]["N"]
    for shape in ((B + 1, N, 3), (0, N, 3), (5, N + 1, 3)):
        with pytest.raises(ValueError):
            tr.step(torch.zeros(shape))
    tr.world = 2      # data parallel without a process group: only the short batch is refused
    with pytest.raises(NotImplementedError):
        tr.step(batch(name, 5, seed=91))
    with pytest.raises(NotImplementedError):
        tr.run_epoch([batch(name, B, seed=92), batch(name, 5, seed=91)])


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_partial_steps_allocate_no_device_memory(graph):
    name, B = "default_b257", 257
    tr = make_trainer(name, B, "bf16", graph, partial=True)
    xf, xs, xt = batch(name, B, seed=100), batch(name, 31, seed=101), batch(name, 200, seed=102)
    for x in (xf, xs, xt):
        tr.step(x)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    for x in (xs, xf, xt, xs, xs):
        tr.step(x)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before


@pytest.mark.gpu
def test_launch_accounting_per_size():
    name, B = "default_b257", 257
    tr = make_trainer(name, B, "bf16", partial=True)
    def counted(t, x):
        before = ops.LAUNCHES["count"]
        t.step(x)
        return ops.LAUNCHES["count"] - before

    for Bp in (B, 64, 3, 64):
        x = batch(name, Bp, seed=110 + Bp)
        fresh = make_trainer(name, Bp, "bf16")
        counted(tr, x)
        counted(fresh, x)
        assert counted(tr, x) == counted(fresh, x) == fresh.launches_per_step == tr.launches_per_step
