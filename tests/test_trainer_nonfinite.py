"""The non-finite step guard of the fused trainer (``GNNAETrainer(nonfinite="skip" | "raise")``) and the non-finite input guards of the
EMD and assignment solvers.  CPU: the keyword check, and the data-parallel decision (gloo, two ranks: a NaN flag element of one rank
and a finite gradient of the other sum to a buffer both ranks skip).  GPU: a trainer that sees [b1, bad, b2] ends bitwise where one
that saw [b1, b2] ends (NaN, Inf and overflowing inputs; every loss; two latent maps; graph and eager; four optimisers; bf16), the
epoch loop, a short last batch, and the solvers' outputs on batches with non-finite jets against runs on the finite jets alone."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from golden_cases import CASES, make_params
from gnn_jet_autoencoder_b200 import EMDLoss, _lib, ops
from gnn_jet_autoencoder_b200.trainer import GNNAETrainer, allreduce_flat_, nonfinite_mode, synthetic_jets

DEV = "cuda"

NF_CASES = {"mean": dict(CASES["default_b257"], B=64), "local_mix": dict(CASES["local_mix_us_n8"], B=37)}

LOSSES = {
    "chamfer": lambda: dict(loss_choice="chamfer"),
    "mse": lambda: dict(loss_choice="mse"),
    "emd_sum": lambda: dict(loss_choice="emd", emd_loss=EMDLoss(polar_coord=False, reduction="sum")),
    "hungarian_abs_cartesian": lambda: dict(loss_choice="hungarian"),
    "hungarian_rel_polar": lambda: dict(loss_choice="hungarian", hungarian_abs_coord=False, hungarian_polar_coord=True),
}


def make_trainer(name="mean", loss="chamfer", nonfinite="skip", graph=True, optimizer="adam", precision="fp32", batch_size=None,
                 partial=False):
    from gnn_jet_autoencoder_b200 import Decoder, Encoder
    case = NF_CASES[name]
    ep, dp = make_params(case)
    enc = Encoder(**case["enc"], device=DEV, precision=precision)
    dec = Decoder(**case["dec"], device=DEV, precision=precision)
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in ep.items()})
    dec.load_state_dict({k: torch.from_numpy(v) for k, v in dp.items()})
    return GNNAETrainer(enc, dec, batch_size=batch_size or case["B"], lr=1e-3, encoder_metric=case["metric"],
                        decoder_metric=case["metric"], use_cuda_graph=graph, optimizer=optimizer, nonfinite=nonfinite,
                        partial_batches=partial, **LOSSES[loss]())


def batch(name, seed, jets=None):
    case = NF_CASES[name]
    return torch.from_numpy(synthetic_jets(jets or case["B"], case["N"], seed=seed)).pin_memory()


def spoil(x, kind):
    """A copy of batch ``x`` with one bad value: a NaN, an Inf, or a jet of finite inputs so large (1e30) that the network and the
    loss overflow."""
    y = x.clone()
    if kind == "nan":
        y[3 % y.shape[0], 2, 1] = float("nan")
    elif kind == "inf":
        y[5 % y.shape[0], 0, 0] = float("inf")
    else:
        y[0] = 1e30
    return y.pin_memory()


def assert_same_state(a, b, grad=True):
    """Parameters and moments bitwise equal, and the gradient of the last step unless that step was a skipped one (its gradient is
    the non-finite one)."""
    torch.cuda.synchronize()
    for attr in ("flat", "exp_avg", "exp_avg_sq") + (("grad",) if grad else ()):
        assert torch.equal(getattr(a, attr), getattr(b, attr)), attr


def check_skip_equivalence(name, loss, bad, graph=True, optimizer="adam", precision="fp32"):
    """[b1, bad, b2] on a "skip" trainer equals [b1, b2] on another, bit for bit; the skipped step returns a non-finite loss."""
    b1, b2 = batch(name, 11), batch(name, 12)
    tr_a = make_trainer(name, loss, "skip", graph, optimizer, precision)
    tr_b = make_trainer(name, loss, "skip", graph, optimizer, precision)
    la = [tr_a.step(b1), tr_a.step(spoil(b1, bad)), tr_a.step(b2)]
    lb = [tr_b.step(b1), tr_b.step(b2)]
    assert not np.isfinite(la[1])
    assert la[0] == lb[0] and la[2] == lb[1]
    assert_same_state(tr_a, tr_b)
    assert tr_a.nonfinite_steps == 1 and tr_b.nonfinite_steps == 0
    assert tr_a.step_count == 3 and tr_a.applied_steps == tr_b.applied_steps == 2
    return tr_a, tr_b, (b1, b2)


# ---------------------------------------------------------------- CPU

def test_nonfinite_keyword_is_checked():
    assert [nonfinite_mode(m) for m in ("ignore", "skip", "raise", "SKIP")] == ["ignore", "skip", "raise", "skip"]
    for bad in ("warn", "", None, True):
        with pytest.raises(ValueError, match="nonfinite must be one of"):
            nonfinite_mode(bad)


def _decide(buf):
    """The decision gj_nonfinite_check takes on the device: skip if any element of the all-reduced buffer is not finite."""
    return not bool(torch.isfinite(buf).all())


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n = 1000
    g = torch.linspace(-1.0, 1.0, n + 1, dtype=torch.float32) * (rank + 1)
    decisions = []
    # (rank whose flag element is NaN, rank whose gradient holds an Inf): the flag of a non-finite local loss, a non-finite local
    # gradient, both, and neither
    for nan_rank, inf_rank in ((0, None), (None, 1), (1, 0), (None, None)):
        buf = g.clone()
        buf[n] = float("nan") if rank == nan_rank else 0.0
        if rank == inf_rank:
            buf[17] = float("inf")
        allreduce_flat_(buf)
        decisions.append(_decide(buf))
    np.save(os.path.join(out_dir, f"decisions{rank}.npy"), np.array(decisions))
    dist.destroy_process_group()


def test_allreduced_flag_makes_every_rank_skip(tmp_path):
    import torch.multiprocessing as mp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    d0, d1 = (np.load(tmp_path / f"decisions{r}.npy").tolist() for r in (0, 1))
    assert d0 == d1 == [True, True, True, False]


# ---------------------------------------------------------------- GPU: the trainer

@pytest.mark.gpu
@pytest.mark.parametrize("config", [("mean", True), ("local_mix", False)], ids=["mean-graph", "local_mix-eager"])
@pytest.mark.parametrize("bad", ["nan", "inf", "huge"])
@pytest.mark.parametrize("loss", sorted(LOSSES))
def test_skipped_step_leaves_no_trace(loss, bad, config):
    name, graph = config
    check_skip_equivalence(name, loss, bad, graph)


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["rmsprop", "adagrad", "sgd"])
def test_skip_with_the_other_optimisers(optimizer):
    tr_a, _, (b1, b2) = check_skip_equivalence("mean", "chamfer", "nan", optimizer=optimizer)
    assert tr_a.applied_steps == 2      # the guarded kernels count applied updates for every optimiser


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_skip_equals_ignore_on_finite_batches(graph):
    """The guarded optimisers apply the unguarded kernels' update: on finite data "skip" and "ignore" train alike, bit for bit."""
    xs = [batch("mean", 20 + k) for k in range(3)]
    tr_s, tr_i = make_trainer(nonfinite="skip", graph=graph), make_trainer(nonfinite="ignore", graph=graph)
    assert [tr_s.step(x) for x in xs] == [tr_i.step(x) for x in xs]
    assert_same_state(tr_s, tr_i)
    assert tr_i.grad_buffer.numel() == tr_i.grad.numel() == tr_s.grad_buffer.numel() - 1
    assert tr_s.applied_steps == tr_i.applied_steps == tr_i.step_count == 3
    if graph:
        assert tr_s.launches_per_step == tr_i.launches_per_step + 2


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("loss", ["chamfer", "hungarian_abs_cartesian"])
def test_raise_mode_raises_with_the_state_kept(loss, graph):
    b1, b2 = batch("mean", 11), batch("mean", 12)
    tr_a, tr_b = make_trainer(loss=loss, nonfinite="raise", graph=graph), make_trainer(loss=loss, nonfinite="raise", graph=graph)
    tr_a.step(b1)
    with pytest.raises(FloatingPointError, match="skipped"):
        tr_a.step(spoil(b1, "nan"))
    tr_a.step(b2)
    tr_b.step(b1)
    tr_b.step(b2)
    assert_same_state(tr_a, tr_b)
    assert tr_a.nonfinite_steps == 1


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_run_epoch_skips_and_names_the_bad_batches(graph):
    b1, b2 = batch("mean", 31), batch("mean", 32)
    epoch = [b1, spoil(b1, "nan"), b2, spoil(b2, "huge")]
    tr_loop = make_trainer(graph=graph)
    losses = [tr_loop.step(b1), tr_loop.step(b2)]
    tr = make_trainer(graph=graph)
    avg, recons, targets, latents = tr.run_epoch(epoch, is_train=True)
    assert tr.last_epoch_nonfinite == [1, 3] and tr.nonfinite_steps == 2
    assert avg == sum(losses) / 2
    assert recons.shape[0] == targets.shape[0] == latents.shape[0] == 4 * b1.shape[0]
    torch.testing.assert_close(targets, torch.cat(epoch), rtol=0, atol=0, equal_nan=True)
    assert_same_state(tr, tr_loop, grad=False)
    assert tr.applied_steps == 2 and tr.step_count == 4
    # validation records the flag only
    before = tr.flat.clone()
    vavg, _, _, _ = tr.run_epoch([b1, spoil(b2, "inf"), b2], is_train=False)
    assert tr.last_epoch_nonfinite == [1] and not np.isfinite(vavg)
    assert torch.equal(tr.flat, before) and tr.nonfinite_steps == 2
    # an epoch in which every update was skipped raises
    with pytest.raises(FloatingPointError, match=r"\[0, 1\] of 2"):
        tr.run_epoch([spoil(b1, "inf"), spoil(b2, "nan")])
    assert torch.equal(tr.flat, before)
    # "raise": the same updates, then the error naming both batches
    tr_r = make_trainer(nonfinite="raise", graph=graph)
    with pytest.raises(FloatingPointError, match=r"\[1, 3\]"):
        tr_r.run_epoch(epoch, is_train=True)
    assert_same_state(tr_r, tr_loop, grad=False)


@pytest.mark.gpu
def test_run_epoch_ignore_is_unchanged_on_finite_batches():
    xs = [batch("mean", 40 + k) for k in range(3)]
    tr_i, tr_s, tr_loop = make_trainer(nonfinite="ignore"), make_trainer(nonfinite="skip"), make_trainer(nonfinite="ignore")
    for tr in (tr_i, tr_s, tr_loop):      # the first step captures the graph (and counts its eager warm-up launches)
        tr.step(xs[0])
    xs = xs[1:]
    losses = [tr_loop.step(x) for x in xs]
    before = ops.LAUNCHES["count"]
    avg_i = tr_i.run_epoch(xs, collect=False)[0]
    launches_i = ops.LAUNCHES["count"] - before
    before = ops.LAUNCHES["count"]
    avg_s = tr_s.run_epoch(xs, collect=False)[0]
    launches_s = ops.LAUNCHES["count"] - before
    assert avg_i == avg_s == sum(losses) / 2
    assert launches_i == 2 * tr_i.launches_per_step and launches_s == launches_i + 2 * 2
    assert tr_i.last_epoch_nonfinite == [] and tr_s.last_epoch_nonfinite == []
    assert_same_state(tr_i, tr_loop)
    assert_same_state(tr_s, tr_loop)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", ["chamfer", "emd_sum"])
def test_short_last_batch_is_skipped(loss):
    b1, b2 = batch("mean", 51), batch("mean", 52)
    short = spoil(batch("mean", 53, jets=23), "nan")
    tr_a = make_trainer(loss=loss, partial=True)
    tr_b = make_trainer(loss=loss, partial=True)
    tr_a.step(b1)
    assert not np.isfinite(tr_a.step(short))
    la = tr_a.step(b2)
    tr_b.step(b1)
    assert la == tr_b.step(b2)
    assert_same_state(tr_a, tr_b)
    avg = tr_a.run_epoch([b1, b2, short])[0]
    tr_b.run_epoch([b1, b2])
    assert tr_a.last_epoch_nonfinite == [2] and np.isfinite(avg)
    assert_same_state(tr_a, tr_b, grad=False)


@pytest.mark.gpu
def test_bf16_deterministic_skip():
    prev = ops.set_deterministic(True)
    try:
        check_skip_equivalence("mean", "chamfer", "nan", precision="bf16")
        check_skip_equivalence("mean", "mse", "huge", precision="bf16")
    finally:
        ops.set_deterministic(prev)


# ---------------------------------------------------------------- GPU: the solvers

def _stream():
    return torch.cuda.current_stream().cuda_stream


def _jets(B, N, D, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((B, N, D), generator=g)
    x[..., 0] = x[..., 0].abs() + 0.1
    return x.to(DEV)


# (side, (particle, component), value); component 0 is avoided, because the energy of a 4-vector enters neither the EMD nor the
# Hungarian loss in polar coordinates (such a jet is solved as usual)
BAD_JETS = {1: ("p", (3, 1), float("nan")), 4: ("q", (0, 1), float("inf")), 5: ("p", (7, 2), -float("inf"))}


def _spoiled_pair(B, N, D, seed):
    p, q = _jets(B, N, D, seed), _jets(B, N, D, seed + 1)
    for b, (side, (k, c), v) in BAD_JETS.items():
        (p if side == "p" else q)[b, k, c] = v
    good = [b for b in range(B) if b not in BAD_JETS]
    return p, q, good


def _run_emd(p, q):
    lib = _lib.load()
    B, Np, Nq = p.shape[0], p.shape[1], q.shape[1]
    f64 = dict(device=DEV, dtype=torch.float64)
    out = dict(emd=torch.empty(B, **f64), flow=torch.empty((B, Np, Nq), **f64),
               dp=torch.empty((B, Np, 3), device=DEV, dtype=torch.float32), pot=torch.empty((B, Np + Nq + 2), **f64),
               status=torch.empty(B, device=DEV, dtype=torch.int32))
    _lib.check(lib.gj_emd(B, Np, Nq, p.data_ptr(), q.data_ptr(), 0.8, 1.0, _lib.GJ_EMD_NORM, out["emd"].data_ptr(), out["flow"].data_ptr(),
                          out["dp"].data_ptr(), out["pot"].data_ptr(), out["status"].data_ptr(), None, 0, _stream()), "gj_emd")
    return out


@pytest.mark.gpu
def test_emd_solver_skips_nonfinite_jets():
    from gnn_jet_autoencoder_b200 import anomaly
    p, q, good = _spoiled_pair(8, 20, 3, seed=5)
    q = q[:, :17].contiguous()
    got = _run_emd(p, q)
    alone = _run_emd(p[good].contiguous(), q[good].contiguous())
    for k, v in alone.items():
        assert torch.equal(got[k][good], v), k
    bad = sorted(BAD_JETS)
    assert got["status"][bad].tolist() == [2] * len(bad) and (alone["status"] == 0).all()
    assert torch.isnan(got["emd"][bad]).all() and torch.isnan(got["pot"][bad]).all()
    assert not got["flow"][bad].any() and not got["dp"][bad].any()
    with pytest.raises(ValueError, match=r"jet\(s\) \[1, 4, 5\]"):
        anomaly.emd(p, q)
    with pytest.raises(ValueError, match=r"jet\(s\) \[2, 3\]"):      # numbered in the whole input when walked in batches
        anomaly.emd(p[2:], q[2:], batch_size=2)


def _run_emd_loss(p, q):
    lib = _lib.load()
    B, N, D = p.shape
    nbytes = int(lib.gj_emd_loss_workspace(B, N))
    ws = torch.zeros(max(nbytes, 1), dtype=torch.uint8, device=DEV)
    terms = torch.empty(3, device=DEV)
    failed = torch.empty(1, device=DEV)
    dp = torch.empty_like(p)
    _lib.check(lib.gj_emd_loss(B, N, D, _lib.GJ_EMD_COORDS_CARTESIAN, p.data_ptr(), q.data_ptr(), 1.0, 1.0, 0, 0.5, terms.data_ptr(),
                               failed.data_ptr(), dp.data_ptr(), ws.data_ptr(), nbytes, _stream()), "gj_emd_loss")
    jet = ws[:8 * B].view(torch.float64)
    status = ws[8 * B:12 * B].view(torch.int32)
    return terms, failed, dp, jet, status


@pytest.mark.gpu
def test_emd_loss_skips_nonfinite_jets():
    p, q, good = _spoiled_pair(8, 24, 4, seed=7)
    terms, failed, dp, jet, status = _run_emd_loss(p, q)
    t_a, f_a, dp_a, jet_a, st_a = _run_emd_loss(p[good].contiguous(), q[good].contiguous())
    assert torch.equal(dp[good], dp_a) and torch.equal(jet[good], jet_a) and torch.equal(status[good], st_a)
    bad = sorted(BAD_JETS)
    assert status[bad].tolist() == [2] * len(bad) and torch.isnan(jet[bad]).all() and not dp[bad].any()
    assert torch.isnan(terms[0]) and torch.isnan(terms[2]) and float(failed) == 0.0 and float(f_a) == 0.0
    assert torch.isfinite(t_a).all()


@pytest.mark.gpu
@pytest.mark.parametrize("lorentz", [0, 1])
def test_assignment_skips_nonfinite_jets(lorentz):
    lib = _lib.load()
    p, q, good = _spoiled_pair(8, 30, 4, seed=9)
    p[6] = 1e30      # finite, but every cost overflows
    good.remove(6)

    def run(a, b):
        B, N, D = a.shape
        match = torch.empty((B, N), device=DEV, dtype=torch.int32)
        total = torch.empty(B, device=DEV)
        _lib.check(lib.gj_assignment(B, N, D, lorentz, a.data_ptr(), b.data_ptr(), match.data_ptr(), total.data_ptr(), _stream()),
                   "gj_assignment")
        return match, total

    match, total = run(p, q)
    m_a, t_a = run(p[good].contiguous(), q[good].contiguous())
    assert torch.equal(match[good], m_a) and torch.equal(total[good], t_a)
    bad = sorted(BAD_JETS) + [6]
    assert (match[bad] == torch.arange(30, device=DEV, dtype=torch.int32)).all() and torch.isnan(total[bad]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("coords", [_lib.GJ_HMSE_ABS_CARTESIAN, _lib.GJ_HMSE_REL_POLAR])
def test_hungarian_loss_skips_nonfinite_jets(coords):
    lib = _lib.load()
    p, q, good = _spoiled_pair(8, 30, 4, seed=11)

    def run(a, b):
        B, N, D = a.shape
        nbytes = int(lib.gj_hungarian_mse_loss_workspace(B, N))
        ws = torch.zeros(max(nbytes, 8), dtype=torch.uint8, device=DEV)
        terms, dp = torch.empty(3, device=DEV), torch.empty_like(a)
        match = torch.empty((B, N), device=DEV, dtype=torch.int32)
        _lib.check(lib.gj_hungarian_mse_loss(B, N, D, coords, a.data_ptr(), b.data_ptr(), 0.25, terms.data_ptr(), dp.data_ptr(),
                                             match.data_ptr(), ws.data_ptr(), nbytes, _stream()), "gj_hungarian_mse_loss")
        return terms, dp, match, ws[:8 * B].view(torch.float64)

    terms, dp, match, jet = run(p, q)
    t_a, dp_a, m_a, jet_a = run(p[good].contiguous(), q[good].contiguous())
    assert torch.equal(dp[good], dp_a) and torch.equal(match[good], m_a) and torch.equal(jet[good], jet_a)
    bad = sorted(BAD_JETS)
    assert (match[bad] == torch.arange(30, device=DEV, dtype=torch.int32)).all()
    assert torch.isnan(jet[bad]).all() and not dp[bad].any() and torch.isnan(terms).any() and torch.isfinite(t_a).all()
