"""The Hungarian-matched MSE of the fused training step: ``gj_hungarian_mse_loss``'s header entry and host-side argument checks
(CPU), and on the GPU the kernel against ``HungarianMSELoss`` + autograd in all four coordinate modes, its matching against
``anomaly.assignment``, ``GNNAETrainer(loss_choice="hungarian")`` against the CUDA modules + ``HungarianMSELoss`` + autograd
(gradients, Adam steps, the epoch loop), reproducibility and the bf16 mode."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from golden_cases import CASES, make_input, make_params
from gnn_jet_autoencoder_b200 import _lib
from gnn_jet_autoencoder_b200.trainer import GNNAETrainer, synthetic_jets

DEV = "cuda"

# coords -> (abs_coord, polar_coord) of HungarianMSELoss.forward
MODES = {_lib.GJ_HMSE_ABS_CARTESIAN: (True, False), _lib.GJ_HMSE_ABS_POLAR: (True, True),
         _lib.GJ_HMSE_REL_POLAR: (False, True), _lib.GJ_HMSE_REL_CARTESIAN: (False, False)}


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


def hungarian_loss(p, q, coords, scale):
    """One gj_hungarian_mse_loss call: (terms (3,) host, dp (B, N, D) device, matching (B, N) int64 device, per-jet losses (B,)
    float64 host, read from the workspace)."""
    lib = _lib.load()
    B, N, D = p.shape
    terms = torch.full((3,), float("nan"), device=DEV)
    dp = torch.full_like(p, float("nan"))
    match = torch.full((B, N), -1, dtype=torch.int32, device=DEV)
    nbytes = int(lib.gj_hungarian_mse_loss_workspace(B, N))
    ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=DEV)
    _lib.check(lib.gj_hungarian_mse_loss(B, N, D, coords, p.data_ptr(), q.data_ptr(), scale, terms.data_ptr(), dp.data_ptr(),
                                         match.data_ptr(), ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream),
               "gj_hungarian_mse_loss")
    return terms.cpu(), dp, match.long(), ws[:8 * B].view(torch.float64).cpu().numpy()


# ---------------------------------------------------------------- CPU

def test_header_declares_the_hungarian_loss_entry_points():
    header = open(os.path.join(ROOT, "include", "gnnjet_b200.h")).read()
    assert re.search(r"\bint gj_hungarian_mse_loss\(", header) and re.search(r"\bsize_t gj_hungarian_mse_loss_workspace\(", header)
    for name, value in (("GJ_HMSE_ABS_CARTESIAN", 0), ("GJ_HMSE_ABS_POLAR", 1), ("GJ_HMSE_REL_POLAR", 2), ("GJ_HMSE_REL_CARTESIAN", 3)):
        assert re.search(rf"#define {name} {value}\b", header), name
        assert getattr(_lib, name) == value


def test_gj_hungarian_mse_loss_rejects_bad_arguments_on_the_host():
    """Argument checks happen before any device work (fake device pointers are never dereferenced)."""
    lib = _lib.load()
    P = 256
    assert lib.gj_hungarian_mse_loss_workspace(64, 30) >= 64 * 8

    def call(batch=4, n=30, dim=3, coords=_lib.GJ_HMSE_ABS_CARTESIAN, ws_bytes=None, terms=P):
        ws_bytes = lib.gj_hungarian_mse_loss_workspace(batch, n) if ws_bytes is None else ws_bytes
        return lib.gj_hungarian_mse_loss(batch, n, dim, coords, P, P, 1.0, terms, P, None, P, ws_bytes, None)

    for kw, msg in (({"n": 0}, "particles per jet <= 220"), ({"n": 221}, "particles per jet <= 220"),
                    ({"batch": -1}, "particles per jet <= 220"), ({"dim": 2}, "features per particle"),
                    ({"dim": 5}, "features per particle"), ({"coords": 4}, "unknown coordinates"),
                    ({"coords": -1}, "unknown coordinates"), ({"ws_bytes": 4 * 8 - 1}, "workspace too small"),
                    ({"terms": None}, "null pointer")):
        assert call(**kw) != 0, kw
        assert msg in _lib.last_error(), (kw, _lib.last_error())


# ---------------------------------------------------------------- GPU: the kernel

def _kernel_order_sum(e):
    """The fixed summation order of gj_hungarian_mse_loss's second launch: 256 strided partial sums, a shuffle tree per warp, the
    8 warps in order."""
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


def on_grid(x, bits):
    """x rounded to multiples of 2^-bits: where every partial sum of a jet fits the fp32 mantissa, the target jet's sum (the axis of
    the relative coordinates) is exact in any order, so the kernel's and torch's axes agree bit for bit."""
    return (np.round(np.asarray(x, np.float64) * 2.0 ** bits) / 2.0 ** bits).astype(np.float32)


def _jets(kind, B, N, D, seed):
    if kind == "random":
        return on_grid(np.random.default_rng(seed).normal(0.0, 1.0, (B, N, D)), 10)
    x = synthetic_jets(B, N, seed=seed)       # zero-padded [pt, eta, phi]; as 4-vectors with E = |x|
    if D == 4:
        x = np.concatenate([np.linalg.norm(x, axis=-1, keepdims=True), x], axis=-1)
    return on_grid(x, 14)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["random", "synthetic"])
@pytest.mark.parametrize("N", [1, 2, 30, 33, 150])
@pytest.mark.parametrize("D", [3, 4])
@pytest.mark.parametrize("coords", sorted(MODES))
def test_kernel_matches_hungarian_mse_loss_autograd(coords, D, N, kind):
    from gnn_jet_autoencoder_b200 import HungarianMSELoss, anomaly
    from gnn_jet_autoencoder_b200.losses import hungarian_preprocess
    abs_coord, polar = MODES[coords]
    B = 16 if N == 150 else 64
    p = torch.from_numpy(_jets(kind, B, N, D, 40 + N + D)).to(DEV)
    q = torch.from_numpy(_jets(kind, B, N, D, 90 + N + D)).to(DEV)
    d_loss = D if coords == _lib.GJ_HMSE_ABS_CARTESIAN else 3
    scale = 1.0 / (B * N * d_loss)
    terms, dp, match, jet = hungarian_loss(p, q, coords, scale)
    grad_tol = 1e-6 if abs_coord else 1e-5

    # the module and autograd
    pg = p.clone().requires_grad_()
    loss = HungarianMSELoss()(pg, q, abs_coord=abs_coord, polar_coord=polar)
    loss.backward()
    assert abs(terms[2].item() - loss.item()) <= 1e-6 * abs(loss.item())
    assert rel(dp.cpu().numpy(), pg.grad.cpu().numpy()) <= grad_tol
    if D == 4 and coords != _lib.GJ_HMSE_ABS_CARTESIAN:
        assert torch.all(dp[..., 0] == 0)

    # the matching
    r, t = hungarian_preprocess(p, q, abs_coord=abs_coord, polar_coord=polar)
    m_ref, total_ref = anomaly.assignment(r, t)
    assert all(sorted(row) == list(range(N)) for row in match.cpu().tolist())
    if abs_coord:
        assert torch.equal(match, m_ref)
    else:       # the target jet's sum may be ordered differently from torch's: the matching is optimal, ties may differ
        t_matched = torch.gather(t, 1, match.unsqueeze(-1).expand(-1, -1, t.shape[-1]))
        total = (r.double() - t_matched.double()).norm(dim=-1).sum(-1)
        assert np.allclose(total.cpu().numpy(), total_ref.double().cpu().numpy(), rtol=1e-5, atol=1e-5)

    # autograd through a gather with the kernel's own matching: the same loss and gradient
    pg2 = p.clone().requires_grad_()
    r2, t2 = hungarian_preprocess(pg2, q, abs_coord=abs_coord, polar_coord=polar)
    shuffled = torch.gather(r2, 1, match.unsqueeze(-1).expand(-1, -1, r2.shape[-1]))
    loss2 = torch.nn.functional.mse_loss(shuffled, t2)
    loss2.backward()
    assert abs(terms[2].item() - loss2.item()) <= 1e-6 * abs(loss2.item())
    assert rel(dp.cpu().numpy(), pg2.grad.cpu().numpy()) <= grad_tol

    # the per-jet values and their fixed-order sum
    want_jet = ((shuffled.detach().double() - t2.double()) ** 2).sum(dim=(1, 2)).cpu().numpy()
    assert np.allclose(jet, want_jet, rtol=1e-5, atol=1e-12)
    assert terms[0].item() == np.float32(_kernel_order_sum(jet))
    scale32 = float(np.float32(scale))        # the C-ABI takes scale as a float
    assert terms[1].item() == 0.0 and terms[2].item() == np.float32(scale32 * _kernel_order_sum(jet))


@pytest.mark.gpu
def test_kernel_is_reproducible_and_scale_only_scales():
    p = torch.from_numpy(_jets("random", 512, 30, 4, 3)).to(DEV)
    q = torch.from_numpy(_jets("random", 512, 30, 4, 4)).to(DEV)
    coords = _lib.GJ_HMSE_REL_CARTESIAN
    t1, dp1, m1, j1 = hungarian_loss(p, q, coords, 1.0)
    t2, dp2, m2, j2 = hungarian_loss(p, q, coords, 1.0)
    assert torch.equal(t1, t2) and torch.equal(dp1, dp2) and torch.equal(m1, m2) and np.array_equal(j1, j2)
    t3, dp3, m3, _ = hungarian_loss(p, q, coords, 0.25)
    assert t3[0].item() == t1[0].item() and torch.equal(m3, m1)
    assert rel(dp3.cpu().numpy(), 0.25 * dp1.cpu().numpy()) <= 1e-7


# ---------------------------------------------------------------- GPU: the trainer

def _module_hungarian(enc, dec, x, case, abs_coord, polar):
    """Reference loop: CUDA modules, the polar clamp of utils/train.py:55-65, HungarianMSELoss, autograd."""
    from gnn_jet_autoencoder_b200 import HungarianMSELoss
    z = enc(x, metric=case["metric"])
    y = dec(z, metric=case["metric"])
    if case["polar_coord"]:
        y = torch.cat([torch.clamp(y[..., :1], min=1e-16), y[..., 1:]], dim=-1)
    return HungarianMSELoss()(y, x, abs_coord=abs_coord, polar_coord=polar)


def _named_module_grads(enc, dec):
    return {**{"encoder." + k: p.grad for k, p in enc.named_parameters()}, **{"decoder." + k: p.grad for k, p in dec.named_parameters()}}


def _trainer(enc, dec, case, abs_coord=True, polar=False, **kw):
    return GNNAETrainer(enc, dec, batch_size=case["B"], encoder_metric=case["metric"], decoder_metric=case["metric"],
                        loss_choice="hungarian", polar_coord=case["polar_coord"], hungarian_abs_coord=abs_coord,
                        hungarian_polar_coord=polar, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["default_n30", "local_mix_us_n8", "polar3_n6", "mink_n6"])
@pytest.mark.parametrize("coords", sorted(MODES))
@pytest.mark.parametrize("graph", [False, True])
def test_trainer_hungarian_gradients_match_the_module_path(models, name, coords, graph):
    abs_coord, polar = MODES[coords]
    case = CASES[name]
    x = torch.from_numpy(on_grid(make_input(case), 16)).to(DEV)
    enc, dec = models(name)
    loss = _module_hungarian(enc, dec, x, case, abs_coord, polar)
    loss.backward()
    ref = _named_module_grads(enc, dec)
    enc2, dec2 = models(name)
    tr = _trainer(enc2, dec2, case, abs_coord, polar, l1_lambda=0.0, use_cuda_graph=graph)
    tr.load_batch(x)
    tr.compute_gradients()
    tr.compute_gradients()      # second call replays the graph / re-runs: results must not accumulate
    torch.cuda.synchronize()
    got = tr.named_gradients()
    names = sorted(ref)
    assert rel(torch.cat([got[k].flatten() for k in names]).cpu().numpy(), torch.cat([ref[k].flatten() for k in names]).cpu().numpy()) <= 1e-5
    stats = tr.stats.cpu().numpy()
    assert stats[1] == 0.0 and stats[5] == 0.0
    assert abs(tr.loss_from_stats(stats) - loss.item()) <= 1e-6 * abs(loss.item())


@pytest.mark.gpu
def test_trainer_hungarian_adam_steps_match_torch(models):
    case = CASES["trainsh_n30"]
    lr = 1e-3
    x = torch.from_numpy(make_input(case)).float().to(DEV)
    enc, dec = models("trainsh_n30")
    opt = torch.optim.Adam(list(enc.parameters()) + list(dec.parameters()), lr=lr, betas=(0.9, 0.999), eps=1e-8)
    enc2, dec2 = models("trainsh_n30")
    tr = _trainer(enc2, dec2, case, lr=lr, l1_lambda=0.0, use_cuda_graph=True)
    xp = x.cpu().pin_memory()
    for _ in range(3):
        opt.zero_grad()
        loss = _module_hungarian(enc, dec, x, case, True, False)
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
def test_trainer_hungarian_run_epoch_equals_the_per_batch_loop(models, graph):
    case = CASES["trainsh_n30"]
    rng = np.random.default_rng(5)
    batches = [torch.from_numpy(make_input(case) * (1.0 + 0.1 * i) + rng.normal(0, 1e-3, make_input(case).shape)).float().pin_memory()
               for i in range(3)]
    enc_a, dec_a = models("trainsh_n30")
    enc_b, dec_b = models("trainsh_n30")
    tr_a = _trainer(enc_a, dec_a, case, False, True, lr=1e-3, use_cuda_graph=graph)
    tr_b = _trainer(enc_b, dec_b, case, False, True, lr=1e-3, use_cuda_graph=graph)
    losses, rec = [], []
    for x in batches:
        losses.append(tr_a.step(x))
        rec.append(tr_a.recon.cpu().clone())
    avg, recons, _, _ = tr_b.run_epoch(batches, is_train=True)
    assert avg == sum(losses) / 3
    assert torch.equal(recons, torch.cat(rec))
    assert torch.equal(tr_a.flat, tr_b.flat)
    before = tr_b.flat.clone()
    vavg, _, _, _ = tr_b.run_epoch([b.to(DEV) for b in batches], is_train=False)
    assert torch.equal(tr_b.flat, before)
    vals = []
    for x in batches:
        tr_a.forward_only(x)
        tr_a._loss(torch.cuda.current_stream().cuda_stream)
        vals.append(tr_a.loss_from_stats(tr_a.stats.cpu()))
    assert vavg == sum(vals) / 3


@pytest.mark.gpu
def test_trainer_hungarian_is_reproducible_at_full_size_and_runs_in_bf16(models):
    B, N = 4096, 30
    x = torch.from_numpy(synthetic_jets(B, N, seed=7))
    out = {}
    for precision in ("fp32", "bf16"):
        enc, dec = models("default_n30", precision)
        tr = GNNAETrainer(enc, dec, batch_size=B, loss_choice="hungarian_mse", hungarian_polar_coord=True)
        tr.load_batch(x)
        tr.compute_gradients()
        g1, s1 = tr.grad.clone(), tr.stats.clone()
        tr.compute_gradients()
        torch.cuda.synchronize()
        if precision == "fp32":
            assert torch.equal(tr.grad, g1) and torch.equal(tr.stats, s1)
        assert torch.isfinite(tr.grad).all()
        out[precision] = tr.loss_from_stats(tr.stats.cpu())
    assert abs(out["bf16"] - out["fp32"]) <= 2e-2 * abs(out["fp32"])
    # N = 150, one step
    enc, dec = models("default_n30", "bf16", num_nodes=150)
    tr = GNNAETrainer(enc, dec, batch_size=256, loss_choice="HungarianMSELoss")
    loss = tr.step(torch.from_numpy(synthetic_jets(256, 150, seed=8)).pin_memory())
    assert np.isfinite(loss) and torch.isfinite(tr.grad).all() and torch.isfinite(tr.flat).all()


@pytest.mark.gpu
def test_trainer_hungarian_constructor_errors(models):
    enc, dec = models("n2")
    with pytest.raises(NotImplementedError):
        GNNAETrainer(enc, dec, batch_size=4, loss_choice="hybrid")
    enc_big, dec_big = models("n2", num_nodes=221)
    with pytest.raises(ValueError, match="220"):
        GNNAETrainer(enc_big, dec_big, batch_size=2, loss_choice="hungarian")
