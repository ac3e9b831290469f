"""Energy mover's distance: the float64 linear-program oracle against closed forms and the C-ABI's argument checks (CPU), and
the device solver ``gj_emd`` -- ``anomaly.emd`` and ``EMDLoss`` -- against the oracle, an optimality certificate at full
batch size, invariances and finite-difference gradients (GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
import emd_oracle as O
from gnn_jet_autoencoder_b200 import _lib
from gnn_jet_autoencoder_b200.trainer import synthetic_jets

DEV = "cuda"


def _jets(rng, B, N, spread=1.0):
    """Random [pt, eta, phi] jets: pt ~ Exp(1), eta ~ N(0, spread^2), phi uniform in [-pi, pi)."""
    return np.stack([rng.exponential(1.0, (B, N)), rng.normal(0.0, spread, (B, N)), rng.uniform(-np.pi, np.pi, (B, N))],
                    axis=-1).astype(np.float32)


def _oracle(p, q, **kw):
    return np.array([O.emd_lp(p[b], q[b], **kw)[0] for b in range(len(p))])


# ---------------------------------------------------------------- CPU: oracle closed forms, C-ABI checks

def test_oracle_identical_jets_give_zero():
    p = _jets(np.random.default_rng(0), 1, 9)[0]
    for beta in (0.5, 1.0, 2.0):
        for norm in (False, True):
            assert abs(O.emd_lp(p, p, beta=beta, norm=norm)[0]) < 1e-9


@pytest.mark.parametrize("R,beta", [(1.0, 1.0), (0.4, 0.5), (0.4, 2.0)])
def test_oracle_one_particle_against_one_particle(R, beta):
    for w, w2 in ((1.0, 1.0), (2.5, 0.7), (0.3, 4.0)):
        p, q = np.array([[w, 0.1, -0.2]]), np.array([[w2, -0.3, 0.4]])
        theta = np.hypot(0.4, 0.6)
        assert abs(O.emd_lp(p, q, R=R, beta=beta)[0] - (min(w, w2) * (theta / R) ** beta + abs(w - w2))) < 1e-9


def test_oracle_jet_against_an_empty_jet_is_its_total_weight():
    p = _jets(np.random.default_rng(1), 1, 7)[0]
    p[2, 0] = -0.5                                         # negative pt carries no weight
    empty = np.zeros((4, 3))
    want = np.maximum(p[:, 0], 0).sum()
    assert abs(O.emd_lp(p, empty)[0] - want) < 1e-6 and abs(O.emd_lp(empty, p)[0] - want) < 1e-6
    assert O.emd_lp(empty, empty)[0] == 0.0
    assert O.emd_lp(p, empty, norm=True)[0] == 1.0


def test_oracle_normalised_translation_in_eta():
    p = _jets(np.random.default_rng(2), 1, 8)[0].astype(np.float64)
    for R, delta in ((1.0, 0.3), (0.4, -0.25)):
        q = p.copy()
        q[:, 1] += delta
        q[:, 0] *= 3.0                                      # the normalisation removes the scale
        assert abs(O.emd_lp(p, q, R=R, beta=1.0, norm=True)[0] - abs(delta) / R) < 1e-8


@pytest.mark.parametrize("swap", [False, True])
def test_oracle_certificate_accepts_the_lp_optimum_and_rejects_perturbations(swap):
    """linprog's duals (alpha <= 0 rows, beta <= 0 columns, gamma total flow) are potentials of the balanced form: gamma goes to
    the lighter jet's side (u = alpha + gamma, v = beta when W_p <= W_q), the dummy on that side is 1 and the other dummy low
    enough to stay feasible."""
    rng = np.random.default_rng(3)
    p, q = _jets(rng, 1, 6)[0], _jets(rng, 1, 5)[0]          # W_p > W_q
    if swap:
        p, q = q, p
    e, f, (al, be, ga) = O.emd_lp(p, q)
    a, b, C, sa, sb = O.weights_and_cost(p, q)
    assert (sa <= sb) == swap
    if sa <= sb:
        u, v = al + ga, be
        ud, vd = 1.0, min(-1.0, 1.0 - u.max())
    else:
        u, v = al, be + ga
        ud, vd = min(-1.0, 1.0 - v.max()), 1.0
    pot = np.concatenate([u, [ud], v, [vd]])
    cert = O.certify(p, q, f, pot, e)
    assert cert["primal"] < 1e-9 and cert["dual"] < 1e-9 and cert["value"] < 1e-9 and cert["gap"] < 1e-7, cert
    assert O.certify(p, q, 0.9 * f, pot, e)["primal"] > 1e-3              # moves too little
    assert O.certify(p, q, f, pot + np.r_[np.full(len(p) + 1, 0.1), np.zeros(len(q) + 1)], e)["dual"] > 1e-3   # u + v > c
    assert O.certify(p, q, f, pot, 1.01 * e)["value"] > 1e-3


def test_header_declares_the_emd_entry_points():
    header = open(os.path.join(ROOT, "include", "gnnjet_b200.h")).read()
    assert re.search(r"\bint gj_emd\(", header) and re.search(r"\bsize_t gj_emd_workspace\(", header)
    assert "GJ_EMD_NORM" in header and "GJ_EMD_PERIODIC_PHI" in header


def test_gj_emd_rejects_bad_arguments_on_the_host():
    """Argument checks happen before any device work (fake device pointers are never dereferenced)."""
    lib = _lib.load()
    P = 256
    assert lib.gj_emd_workspace(64, 150, 150) == 0

    def call(batch=4, np_=30, nq=30, R=1.0, beta=1.0, flags=0, emd=P):
        return lib.gj_emd(batch, np_, nq, P, P, R, beta, flags, emd, None, None, None, None, None, 0, None)

    for kw, msg in (({"np_": 151}, "particles per jet"), ({"nq": 151}, "particles per jet"), ({"np_": 0}, "particles per jet"),
                    ({"batch": -1}, "particles per jet"), ({"R": 0.0}, "R must be positive"), ({"R": -1.0}, "R must be positive"),
                    ({"R": float("inf")}, "R must be positive"), ({"beta": 0.0}, "beta must be positive"),
                    ({"beta": float("nan")}, "beta must be positive"), ({"flags": 4}, "unknown flags"), ({"emd": None}, "null pointer")):
        assert call(**kw) == 1, kw
        assert msg in _lib.last_error(), (kw, _lib.last_error())
    assert call(batch=0) == 0 and _lib.last_error() == ""      # an empty batch launches nothing


def test_emd_loss_validates_its_options():
    from gnn_jet_autoencoder_b200 import EMDLoss
    with pytest.raises(ValueError):
        EMDLoss(reduction="max")
    with pytest.raises(ValueError):
        EMDLoss(R=0.0)
    with pytest.raises(ValueError):
        EMDLoss(beta=-1.0)


# ---------------------------------------------------------------- GPU: device solver

def _dev_emd(p, q, **kw):
    from gnn_jet_autoencoder_b200 import anomaly
    return anomaly.emd(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV), **kw).cpu().numpy()


def _solve(p, q, R=1.0, beta=1.0, norm=False, periodic_phi=False):
    from gnn_jet_autoencoder_b200.anomaly import _emd_solve
    e, f, _, pot = _emd_solve(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV), R, beta, norm, periodic_phi, want_flow=True,
                              want_potentials=True)
    return e.cpu().numpy(), f.cpu().numpy(), pot.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("np_,nq", [(1, 1), (1, 7), (30, 30), (30, 17), (150, 150)])
def test_emd_matches_linprog(np_, nq):
    """Per-jet EMD within 1e-5 relative (+ 1e-7 absolute) of the float64 linear program, random and synthetic_jets batches,
    over beta, R, norm and periodic phi."""
    rng = np.random.default_rng(np_ * 1000 + nq)
    big = np_ * nq > 2000
    B = 1 if big else 6
    sets = [(_jets(rng, B, np_), _jets(rng, B, nq))]
    sets.append((synthetic_jets(B, np_, seed=np_ + 7), synthetic_jets(B, nq, seed=nq + 11)))
    combos = [(beta, R, norm, per) for beta in (0.5, 1.0, 2.0) for R in (0.4, 1.0) for norm in (False, True) for per in (False, True)]
    if big:      # linprog takes seconds per 150 x 150 jet: every option value, not every combination
        combos = [(0.5, 0.4, False, True), (1.0, 1.0, True, False), (2.0, 0.4, True, True), (1.0, 0.4, False, False)]
    for p, q in sets:
        for beta, R, norm, per in combos:
            kw = dict(R=R, beta=beta, norm=norm, periodic_phi=per)
            got, want = _dev_emd(p, q, **kw), _oracle(p, q, **kw)
            assert got.dtype == np.float64 and got.shape == (B,)
            assert np.all(np.abs(got - want) <= 1e-5 * np.abs(want) + 1e-7), (kw, got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("B,N", [(4096, 30), (256, 150)])
def test_emd_optimality_certificate_at_full_size(B, N):
    """Every jet of a full batch: the returned flow is feasible and moves min(W_p, W_q), the potentials are dual feasible, and
    primal and dual objectives agree to 1e-6 relative (so the EMD is optimal without an LP solver)."""
    rng = np.random.default_rng(B + N)
    p = synthetic_jets(B, N, seed=B + 1)
    q = synthetic_jets(B, N, seed=B + 2)
    q[: B // 2] = _jets(rng, B // 2, N, spread=0.3)        # half with unequal totals
    for kw in (dict(R=0.4, beta=1.0), dict(R=1.0, beta=2.0, norm=True)):
        e, f, pot = _solve(p, q, **kw)
        worst = {"primal": 0.0, "dual": 0.0, "gap": 0.0, "value": 0.0}
        for b in range(B):
            c = O.certify(p[b], q[b], f[b], pot[b], e[b], **kw)
            worst = {k: max(worst[k], c[k]) for k in worst}
        assert worst["primal"] < 1e-9 and worst["dual"] < 1e-6 and worst["gap"] < 1e-6 and worst["value"] < 1e-6, (kw, worst)


@pytest.mark.gpu
def test_emd_invariances():
    """Symmetry in p <-> q, invariance under particle permutations and zero padding, negative pt counted as 0."""
    rng = np.random.default_rng(5)
    B, N = 64, 30
    p, q = _jets(rng, B, N, 0.5), _jets(rng, B, 23, 0.5)
    for kw in (dict(), dict(R=0.4, beta=2.0, norm=True, periodic_phi=True), dict(beta=0.5)):
        base = _dev_emd(p, q, **kw)
        tol = 1e-6 * np.abs(base) + 1e-9
        assert np.all(np.abs(_dev_emd(q, p, **kw) - base) <= tol), kw
        perm_p = p[:, rng.permutation(N)]
        perm_q = q[:, rng.permutation(23)]
        assert np.all(np.abs(_dev_emd(perm_p, perm_q, **kw) - base) <= tol), kw
        pad_p = np.concatenate([p, np.zeros((B, 5, 3), np.float32)], 1)
        pad_q = np.concatenate([np.zeros((B, 9, 3), np.float32), q], 1)
        assert np.all(np.abs(_dev_emd(pad_p, pad_q, **kw) - base) <= tol), kw
        neg = pad_p.copy()
        neg[:, N:, 0] = -rng.uniform(0.1, 1.0, (B, 5))
        neg[:, N:, 1:] = rng.normal(size=(B, 5, 2))
        assert np.all(np.abs(_dev_emd(neg, pad_q, **kw) - base) <= tol), kw


@pytest.mark.gpu
def test_emd_degenerate_problems_converge_and_are_reproducible():
    """Empty jets, duplicated particles and identical jets (ties everywhere) converge to the closed forms; two runs agree
    bitwise."""
    from gnn_jet_autoencoder_b200 import anomaly
    rng = np.random.default_rng(6)
    B, N = 32, 30
    p = _jets(rng, B, N, 0.2)
    p[:, 10:20] = p[:, :10]                                  # duplicated particles
    q = p.copy()
    q[:, :, 0] = np.round(q[:, :, 0] * 4) / 4               # equal weights, many ties
    empty = np.zeros_like(p)
    w = np.maximum(p[..., 0].astype(np.float64), 0).sum(1)
    assert np.allclose(_dev_emd(p, empty), w, rtol=1e-6) and np.allclose(_dev_emd(empty, p), w, rtol=1e-6)
    assert np.all(_dev_emd(empty, empty) == 0.0)
    assert np.all(np.abs(_dev_emd(p, p, beta=0.5)) <= 1e-6 * w)
    assert np.allclose(_dev_emd(p, empty, norm=True), 1.0, rtol=0, atol=1e-12)
    for kw in (dict(), dict(norm=True, beta=2.0)):
        want = _oracle(p[:4], q[:4], **kw)
        got = _dev_emd(p, q, **kw)
        assert np.all(np.abs(got[:4] - want) <= 1e-5 * np.abs(want) + 1e-7)
        a = anomaly.emd(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV), return_flow=True, **kw)
        b = anomaly.emd(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV), return_flow=True, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_emd_flow_output_and_batched_host_path():
    """return_flow gives (B, Np, Nq) float64 flows whose cost reproduces the EMD; a positive batch_size gives host tensors equal
    to one launch; polar_coord=False converts Cartesian 4-vectors like hungarian_preprocess."""
    from gnn_jet_autoencoder_b200 import anomaly
    from gnn_jet_autoencoder_b200.losses import _to_polar
    rng = np.random.default_rng(8)
    p, q = _jets(rng, 40, 12, 0.5), _jets(rng, 40, 9, 0.5)
    pd, qd = torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV)
    e, f = anomaly.emd(pd, qd, R=0.4, return_flow=True)
    assert f.shape == (40, 12, 9) and f.dtype == torch.float64 and e.is_cuda
    a, b, C, sa, sb = O.weights_and_cost(p[3], q[3], R=0.4)
    assert abs(float((f[3].cpu().numpy() * C).sum()) + abs(sa - sb) - float(e[3])) <= 1e-6 * float(e[3])
    eb, fb = anomaly.emd(pd, qd, R=0.4, batch_size=16, return_flow=True)
    assert not eb.is_cuda and torch.equal(eb, e.cpu()) and torch.equal(fb, f.cpu())
    assert torch.equal(anomaly.emd(torch.from_numpy(p), torch.from_numpy(q), R=0.4), e.cpu())      # CPU in, CPU out
    cart = rng.normal(size=(5, 10, 4)).astype(np.float32)
    cart2 = rng.normal(size=(5, 8, 4)).astype(np.float32)
    c1, c2 = torch.from_numpy(cart).to(DEV), torch.from_numpy(cart2).to(DEV)
    assert torch.equal(anomaly.emd(c1, c2, polar_coord=False), anomaly.emd(_to_polar(c1), _to_polar(c2)))
    with pytest.raises(ValueError):
        anomaly.emd(c1, c2)                                   # 4-vectors need polar_coord=False
    with pytest.raises(_lib.GnnJetError):
        anomaly.emd(torch.zeros(2, 151, 3, device=DEV), torch.zeros(2, 3, 3, device=DEV))


def _fd_grad(p, q, h=1e-4, **kw):
    g = np.zeros_like(p, dtype=np.float64)
    for i in range(p.shape[0]):
        for k in range(3):
            pp, pm = p.astype(np.float64), p.astype(np.float64)
            pp[i, k] += h
            pm[i, k] -= h
            g[i, k] = (O.emd_lp(pp, q, **kw)[0] - O.emd_lp(pm, q, **kw)[0]) / (2 * h)
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(R=0.4, beta=2.0), dict(beta=0.5, norm=True), dict(R=0.7, beta=1.0, norm=True, periodic_phi=True)])
def test_emd_loss_gradient_matches_finite_differences(kw):
    """EMDLoss backward (the kernel's dp) against central differences of the float64 oracle, all three components, on small
    generic jets (unequal totals, particles well separated)."""
    from gnn_jet_autoencoder_b200 import EMDLoss
    rng = np.random.default_rng(9)
    B, Np, Nq = 3, 5, 6
    p = np.stack([rng.uniform(0.5, 2.0, (B, Np)), rng.normal(0, 1, (B, Np)), rng.uniform(-2.5, 2.5, (B, Np))], -1).astype(np.float32)
    q = np.stack([rng.uniform(0.5, 2.0, (B, Nq)), rng.normal(0, 1, (B, Nq)), rng.uniform(-2.5, 2.5, (B, Nq))], -1).astype(np.float32)
    p[0, 0, 0] = -0.3                                         # clamped: no pt gradient, no weight
    pt = torch.from_numpy(p).to(DEV).requires_grad_(True)
    loss = EMDLoss(**kw)(pt, torch.from_numpy(q).to(DEV))
    loss.backward()
    g = pt.grad.cpu().numpy()
    assert abs(loss.item() - _oracle(p, q, **kw).sum()) <= 1e-5 * abs(loss.item())
    fd = np.stack([_fd_grad(p[b], q[b], **kw) for b in range(B)])
    assert g[0, 0, 0] == 0.0 and fd[0, 0, 0] == 0.0
    assert np.abs(g - fd).max() <= 2e-3 * np.abs(fd).max(), np.abs(g - fd).max()


@pytest.mark.gpu
def test_emd_loss_reductions_and_cartesian_input():
    from gnn_jet_autoencoder_b200 import EMDLoss, anomaly
    rng = np.random.default_rng(10)
    p, q = _jets(rng, 8, 10, 0.5), _jets(rng, 8, 10, 0.5)
    pd, qd = torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV)
    per_jet = anomaly.emd(pd, qd, R=0.4)
    none = EMDLoss(R=0.4, reduction="none")(pd, qd)
    assert none.shape == (8,) and none.dtype == torch.float32 and torch.allclose(none.double(), per_jet, rtol=1e-6)
    assert torch.allclose(EMDLoss(R=0.4)(pd, qd).double(), per_jet.sum(), rtol=1e-6)
    assert torch.allclose(EMDLoss(R=0.4, reduction="mean")(pd, qd).double(), per_jet.mean(), rtol=1e-6)
    # gradient of "mean" is that of "sum" / B; float64 recons get a float64 gradient
    x = pd.double().requires_grad_(True)
    EMDLoss(R=0.4, reduction="mean")(x, qd).backward()
    y = pd.clone().requires_grad_(True)
    EMDLoss(R=0.4)(y, qd).backward()
    assert x.grad.dtype == torch.float64 and torch.allclose(x.grad.float() * 8, y.grad, rtol=1e-5, atol=1e-7)
    # Cartesian 4-vectors: the gradient reaches them through _to_polar
    c = torch.randn(4, 10, 4, device=DEV, generator=torch.Generator(DEV).manual_seed(0)).requires_grad_(True)
    t = torch.randn(4, 7, 4, device=DEV, generator=torch.Generator(DEV).manual_seed(1))
    EMDLoss(polar_coord=False)(c, t).backward()
    assert c.grad.shape == c.shape and torch.isfinite(c.grad).all() and c.grad.abs().sum() > 0
    with pytest.raises(NotImplementedError):
        EMDLoss()(pd, qd.clone().requires_grad_(True))
