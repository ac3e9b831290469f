"""The EMD loss of the fused training step: ``gj_emd_loss``'s host-side argument checks and the trainer's failure guard (CPU), and
on the GPU the kernel against ``gj_emd`` and the torch conversion of ``EMDLoss``, ``GNNAETrainer(loss_choice="emd")`` against
the CUDA modules + ``EMDLoss`` + autograd (gradients, Adam steps, the epoch loop), reproducibility and the bf16 mode."""
import os
import re
import types

import numpy as np
import pytest
import torch

from conftest import ROOT
from golden_cases import CASES, make_input, make_params
from gnn_jet_autoencoder_b200 import _lib
from gnn_jet_autoencoder_b200.trainer import GNNAETrainer, synthetic_jets

DEV = "cuda"


def rel(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


@pytest.fixture
def models():
    """build(name, precision) -> (encoder, decoder) CUDA modules of a golden case with its seeded parameters."""
    def build(name, precision="fp32", **override):
        from gnn_jet_autoencoder_b200 import Decoder, Encoder
        case = CASES[name]
        ep, dp = make_params(case)
        enc = Encoder(**{**case["enc"], **override}, device=DEV, precision=precision)
        dec = Decoder(**{**case["dec"], **override}, device=DEV, precision=precision)
        if not override:
            enc.load_state_dict({k: torch.from_numpy(v) for k, v in ep.items()})
            dec.load_state_dict({k: torch.from_numpy(v) for k, v in dp.items()})
        return enc, dec
    return build


def emd_loss(p, q, coords, R=1.0, beta=1.0, flags=0, scale=1.0):
    """One gj_emd_loss call: (terms (3,) host, failed (float), dp (B, N, D) device)."""
    lib = _lib.load()
    B, N, D = p.shape
    terms = torch.full((3,), float("nan"), device=DEV)
    failed = torch.full((1,), float("nan"), device=DEV)
    dp = torch.full_like(p, float("nan"))
    nbytes = int(lib.gj_emd_loss_workspace(B, N))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=DEV)
    _lib.check(lib.gj_emd_loss(B, N, D, coords, p.data_ptr(), q.data_ptr(), R, beta, flags, scale, terms.data_ptr(), failed.data_ptr(),
                               dp.data_ptr(), ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream), "gj_emd_loss")
    return terms.cpu(), float(failed.item()), dp


# ---------------------------------------------------------------- CPU

def test_header_declares_the_emd_loss_entry_points():
    header = open(os.path.join(ROOT, "include", "gnnjet_b200.h")).read()
    assert re.search(r"\bint gj_emd_loss\(", header) and re.search(r"\bsize_t gj_emd_loss_workspace\(", header)
    assert "GJ_EMD_COORDS_POLAR" in header and "GJ_EMD_COORDS_CARTESIAN" in header


def test_gj_emd_loss_rejects_bad_arguments_on_the_host():
    """Argument checks happen before any device work (fake device pointers are never dereferenced)."""
    lib = _lib.load()
    P = 256
    assert lib.gj_emd_loss_workspace(64, 30) >= 64 * 12

    def call(batch=4, n=30, dim=3, coords=_lib.GJ_EMD_COORDS_POLAR, R=1.0, beta=1.0, flags=0, ws_bytes=None):
        ws_bytes = lib.gj_emd_loss_workspace(batch, n) if ws_bytes is None else ws_bytes
        return lib.gj_emd_loss(batch, n, dim, coords, P, P, R, beta, flags, 1.0, P, P, P, P, ws_bytes, None)

    cart = _lib.GJ_EMD_COORDS_CARTESIAN
    for kw, msg in (({"n": 0}, "particles per jet"), ({"n": 151}, "particles per jet"), ({"batch": -1}, "particles per jet"),
                    ({"dim": 5, "coords": cart}, "features per particle"), ({"dim": 2, "coords": cart}, "features per particle"),
                    ({"dim": 4}, "polar coordinates"), ({"coords": 2}, "unknown coordinates"),
                    ({"R": 0.0}, "R must be positive"), ({"R": -1.0}, "R must be positive"),
                    ({"R": float("inf")}, "R must be positive"), ({"beta": 0.0}, "beta must be positive"),
                    ({"beta": -2.0}, "beta must be positive"), ({"beta": float("nan")}, "beta must be positive"),
                    ({"flags": 4}, "unknown flags"), ({"ws_bytes": 4 * 12 - 1}, "workspace too small")):
        assert call(**kw) != 0, kw
        assert msg in _lib.last_error(), (kw, _lib.last_error())


def test_loss_from_stats_raises_when_the_emd_solver_hit_its_cap():
    holder = types.SimpleNamespace(l1=0.5, l2=0.0)
    row = np.array([3.0, 0.0, 3.0, 2.0, 0.0, 0.0, 0.0, 0.0], np.float32)
    assert GNNAETrainer.loss_from_stats(holder, row) == 4.0
    row[5] = 1.0
    with pytest.raises(RuntimeError, match="did not converge"):
        GNNAETrainer.loss_from_stats(holder, row)


# ---------------------------------------------------------------- GPU: the kernel

def _kernel_order_sum(e):
    """The fixed summation order of gj_emd_loss's second launch: 256 strided partial sums, a shuffle tree per warp, the 8 warps
    in order."""
    part = np.zeros(256)
    for k in range(0, len(e), 256):
        chunk = e[k:k + 256]
        part[:len(chunk)] = part[:len(chunk)] + chunk
    s = part.reshape(8, 32).copy()
    for d in (16, 8, 4, 2, 1):
        s[:, :d] = s[:, :d] + s[:, d:2 * d]
    t = 0.0
    for w in range(8):
        t = t + s[w, 0]
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{}, dict(R=0.4, beta=2.0), dict(R=1.0, beta=0.5, norm=True),
                                dict(R=0.7, beta=1.0, norm=True, periodic_phi=True)])
def test_polar_kernel_equals_gj_emd(kw):
    from gnn_jet_autoencoder_b200.anomaly import _emd_solve
    B = 1000
    p = torch.from_numpy(synthetic_jets(B, 30, seed=11)).to(DEV)
    q = torch.from_numpy(synthetic_jets(B, 30, seed=12)).to(DEV)
    R, beta = kw.get("R", 1.0), kw.get("beta", 1.0)
    norm, periodic = kw.get("norm", False), kw.get("periodic_phi", False)
    e, _, dp_ref, _ = _emd_solve(p, q, R, beta, norm, periodic, want_grad=True)
    flags = (_lib.GJ_EMD_NORM if norm else 0) | (_lib.GJ_EMD_PERIODIC_PHI if periodic else 0)
    terms, failed, dp = emd_loss(p, q, _lib.GJ_EMD_COORDS_POLAR, R, beta, flags)
    assert torch.equal(dp, dp_ref)
    e = e.cpu().numpy()
    assert terms[0].item() == np.float32(_kernel_order_sum(e))
    assert abs(terms[0].item() - e.sum()) <= 1e-6 * e.sum()
    assert terms[1].item() == 0.0 and terms[2].item() == terms[0].item() and failed == 0.0
    # scale multiplies the gradient and terms[2] only
    t2, _, dp2 = emd_loss(p, q, _lib.GJ_EMD_COORDS_POLAR, R, beta, flags, scale=0.25)
    assert t2[0].item() == terms[0].item() and t2[2].item() == np.float32(0.25 * _kernel_order_sum(e))
    assert torch.equal(dp2, dp_ref * 0.25)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [3, 4])
@pytest.mark.parametrize("kw", [{}, dict(R=0.4, beta=2.0, norm=True)])
def test_cartesian_kernel_equals_emd_loss_autograd(D, kw):
    from gnn_jet_autoencoder_b200 import EMDLoss
    rng = np.random.default_rng(20 + D)
    p = torch.from_numpy(rng.normal(0.0, 1.0, (64, 20, D)).astype(np.float32)).to(DEV)
    q = torch.from_numpy(rng.normal(0.0, 1.0, (64, 20, D)).astype(np.float32)).to(DEV)
    pg = p.clone().requires_grad_()
    loss = EMDLoss(polar_coord=False, **kw)(pg, q)
    loss.backward()
    flags = _lib.GJ_EMD_NORM if kw.get("norm") else 0
    terms, failed, dp = emd_loss(p, q, _lib.GJ_EMD_COORDS_CARTESIAN, kw.get("R", 1.0), kw.get("beta", 1.0), flags)
    assert failed == 0.0 and terms[1].item() == 0.0
    assert abs(terms[0].item() - loss.item()) <= 1e-5 * abs(loss.item())
    assert abs(terms[2].item() - loss.item()) <= 1e-5 * abs(loss.item())
    assert rel(dp.cpu().numpy(), pg.grad.cpu().numpy()) <= 1e-5
    if D == 4:
        assert torch.all(dp[..., 0] == 0)


# ---------------------------------------------------------------- GPU: the trainer

def _module_emd(enc, dec, x, case, crit):
    """Reference loop: CUDA modules, the polar clamp of utils/train.py:55-65, EMDLoss, autograd."""
    z = enc(x, metric=case["metric"])
    y = dec(z, metric=case["metric"])
    if case["polar_coord"]:
        y = torch.cat([torch.clamp(y[..., :1], min=1e-16), y[..., 1:]], dim=-1)
    return crit(y, x)


def _named_module_grads(enc, dec):
    return {**{"encoder." + k: p.grad for k, p in enc.named_parameters()}, **{"decoder." + k: p.grad for k, p in dec.named_parameters()}}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["default_n30", "local_mix_us_n8", "polar3_n6", "mink_n6"])
@pytest.mark.parametrize("reduction", ["sum", "mean"])
@pytest.mark.parametrize("graph", [False, True])
def test_trainer_emd_gradients_match_the_module_path(models, name, reduction, graph):
    from gnn_jet_autoencoder_b200 import EMDLoss
    case = CASES[name]
    x = torch.from_numpy(make_input(case)).float().to(DEV)
    enc, dec = models(name)
    crit = EMDLoss(polar_coord=case["polar_coord"], reduction=reduction)
    loss = _module_emd(enc, dec, x, case, crit)
    loss.backward()
    ref = _named_module_grads(enc, dec)
    enc2, dec2 = models(name)
    tr = GNNAETrainer(enc2, dec2, batch_size=case["B"], l1_lambda=0.0, encoder_metric=case["metric"], decoder_metric=case["metric"],
                      use_cuda_graph=graph, loss_choice="emd", polar_coord=case["polar_coord"],
                      emd_loss=EMDLoss(polar_coord=case["polar_coord"], reduction=reduction))
    tr.load_batch(x)
    tr.compute_gradients()
    tr.compute_gradients()      # second call replays the graph / re-runs: results must not accumulate
    torch.cuda.synchronize()
    got = tr.named_gradients()
    names = sorted(ref)
    assert rel(torch.cat([got[k].flatten() for k in names]).cpu().numpy(), torch.cat([ref[k].flatten() for k in names]).cpu().numpy()) <= 1e-5
    stats = tr.stats.cpu().numpy()
    assert stats[5] == 0.0
    assert abs(tr.loss_from_stats(stats) - loss.item()) <= 1e-6 * abs(loss.item())


@pytest.mark.gpu
def test_trainer_emd_adam_steps_match_torch(models):
    from gnn_jet_autoencoder_b200 import EMDLoss
    case = CASES["trainsh_n30"]
    lr = 1e-3
    x = torch.from_numpy(make_input(case)).float().to(DEV)
    enc, dec = models("trainsh_n30")
    crit = EMDLoss(polar_coord=False)
    opt = torch.optim.Adam(list(enc.parameters()) + list(dec.parameters()), lr=lr, betas=(0.9, 0.999), eps=1e-8)
    enc2, dec2 = models("trainsh_n30")
    tr = GNNAETrainer(enc2, dec2, batch_size=case["B"], lr=lr, l1_lambda=0.0, loss_choice="emd", use_cuda_graph=True)
    xp = x.cpu().pin_memory()
    for _ in range(3):
        opt.zero_grad()
        loss = _module_emd(enc, dec, x, case, crit)
        loss.backward()
        opt.step()
        got = tr.step(xp)
        assert abs(got - loss.item()) <= 1e-5 * abs(loss.item())
    for a, b in ((enc, enc2), (dec, dec2)):
        sa, sb = a.state_dict(), b.state_dict()
        for k in sa:
            assert rel(sb[k].cpu().numpy(), sa[k].cpu().numpy()) <= 1e-5, k


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_trainer_emd_run_epoch_equals_the_per_batch_loop(models, graph):
    case = CASES["trainsh_n30"]
    B = case["B"]
    rng = np.random.default_rng(5)
    batches = [torch.from_numpy(make_input(case) * (1.0 + 0.1 * i) + rng.normal(0, 1e-3, make_input(case).shape)).float().pin_memory()
               for i in range(3)]
    enc_a, dec_a = models("trainsh_n30")
    enc_b, dec_b = models("trainsh_n30")
    tr_a = GNNAETrainer(enc_a, dec_a, batch_size=B, lr=1e-3, use_cuda_graph=graph, loss_choice="emd")
    tr_b = GNNAETrainer(enc_b, dec_b, batch_size=B, lr=1e-3, use_cuda_graph=graph, loss_choice="emd")
    losses, rec = [], []
    for x in batches:
        losses.append(tr_a.step(x))
        rec.append(tr_a.recon.cpu().clone())
    avg, recons, _, _ = tr_b.run_epoch(batches, is_train=True)
    assert avg == sum(losses) / 3
    assert torch.equal(recons, torch.cat(rec))
    assert torch.equal(tr_a.flat, tr_b.flat)
    before = tr_b.flat.clone()
    vavg, vrec, _, _ = tr_b.run_epoch([b.to(DEV) for b in batches], is_train=False)
    assert torch.equal(tr_b.flat, before)
    vals = []
    for x in batches:
        tr_a.load_batch(x)
        tr_a.forward_only(x)
        tr_a._loss(torch.cuda.current_stream().cuda_stream)
        vals.append(tr_a.loss_from_stats(tr_a.stats.cpu()))
    assert vavg == sum(vals) / 3


@pytest.mark.gpu
def test_trainer_emd_is_reproducible_at_full_size_and_runs_in_bf16(models):
    from gnn_jet_autoencoder_b200 import EMDLoss
    B, N = 4096, 30
    x = torch.from_numpy(synthetic_jets(B, N, seed=7))
    out = {}
    for precision in ("fp32", "bf16"):
        enc, dec = models("default_n30", precision)
        tr = GNNAETrainer(enc, dec, batch_size=B, loss_choice="emd", polar_coord=True, emd_loss=EMDLoss(polar_coord=True))
        tr.load_batch(x)
        tr.compute_gradients()
        g1, s1 = tr.grad.clone(), tr.stats.clone()
        tr.compute_gradients()
        torch.cuda.synchronize()
        if precision == "fp32":
            assert torch.equal(tr.grad, g1) and torch.equal(tr.stats, s1)
        assert tr.stats[5].item() == 0.0 and torch.isfinite(tr.grad).all()
        out[precision] = tr.loss_from_stats(tr.stats.cpu())
    assert abs(out["bf16"] - out["fp32"]) <= 2e-2 * abs(out["fp32"])


@pytest.mark.gpu
def test_trainer_emd_constructor_errors(models):
    from gnn_jet_autoencoder_b200 import EMDLoss
    enc, dec = models("n2")
    with pytest.raises(ValueError, match="reduction"):
        GNNAETrainer(enc, dec, batch_size=4, loss_choice="emd", emd_loss=EMDLoss(polar_coord=False, reduction="none"))
    with pytest.raises(ValueError, match="polar_coord"):
        GNNAETrainer(enc, dec, batch_size=4, loss_choice="emd", emd_loss=EMDLoss(polar_coord=True))
    with pytest.raises(ValueError, match="polar_coord"):
        GNNAETrainer(enc, dec, batch_size=4, loss_choice="EMD_loss", polar_coord=True, emd_loss=EMDLoss(polar_coord=False))
    with pytest.raises(NotImplementedError):
        GNNAETrainer(enc, dec, batch_size=4, loss_choice="hybrid")
    enc4, dec4 = models("mink_n6")
    with pytest.raises(ValueError, match="3 features"):
        GNNAETrainer(enc4, dec4, batch_size=3, loss_choice="emd", polar_coord=True)
    enc_big, dec_big = models("n2", num_nodes=151)
    with pytest.raises(ValueError, match="150"):
        GNNAETrainer(enc_big, dec_big, batch_size=2, loss_choice="emdloss")
