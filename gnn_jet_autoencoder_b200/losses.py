"""ChamferLoss: drop-in for reference utils/losses/chamfer_loss/chamfer_loss.py on one fused kernel; HungarianMSELoss
(utils/losses/hungarian_mse) with the matching on the device; EMDLoss, the exact energy mover's distance."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops


def _norm_id(p: torch.Tensor, norm_choice: str) -> int:
    """Norm id handed to ``gj_chamfer_fwd_bwd``: 'minkowskian' and 'polar' both evaluate 2*p0^2 - sum p^2
    (distance_sq.py:57-77), anything else is the euclidean square.  The kernel itself forces the PAIRWISE term of
    3-vectors to cartesian (distance_sq.py:43-44) but keeps the requested norm in the jet term, which the reference
    evaluates with ``normsq(jet_p - jet_q, norm_choice=self.loss_norm_choice)`` (chamfer_loss.py:40)."""
    return 1 if str(norm_choice).lower() in ("minkowskian", "polar") else 0


class ChamferLoss(nn.Module):
    """sum_b [sum_i min_j d(p_i,q_j) + sum_j min_i d(p_i,q_j)] + w * sum_b normsq(sum_i p_i - sum_i q_i).

    ``mode="intended"`` (default) returns that value -- what chamfer_loss.py:26-41 computes.
    ``mode="reference"`` reproduces what the reference actually RETURNS: the jet term alone
    (chamfer_loss.py:42 returns ``jet_loss``), and like the reference raises ``UnboundLocalError`` for
    ``jet_features_weight == 0``.  ``last_terms`` holds [chamfer term, jet term, returned value].
    p: reconstructed jets (B,N,D), receives the gradient; q: target jets (B,N',D); D in {3,4}.
    """

    def __init__(self, loss_norm_choice: str = "cartesian", mode: str = "intended"):
        super().__init__()
        if mode not in ("intended", "reference"):
            raise ValueError("mode must be 'intended' or 'reference'")
        self.loss_norm_choice = loss_norm_choice
        self.mode = mode
        self.last_terms = None

    def forward(self, p: torch.Tensor, q: torch.Tensor, jet_features_weight=1):
        self.device = p.device
        if self.mode == "reference":
            if jet_features_weight == 0:
                raise UnboundLocalError("jet_loss referenced before assignment (reference chamfer_loss.py:42)")
            wc, wj = 0.0, 1.0
        else:
            wc, wj = 1.0, float(jet_features_weight)
        q = q.to(device=p.device)
        loss, terms = ops.chamfer_loss(p.float(), q.float(), _norm_id(p, self.loss_norm_choice), wc, wj)
        self.last_terms = terms
        return loss if p.dtype == torch.float32 else loss.to(p.dtype)


_HEPS = 1e-16      # utils/losses/hungarian_mse/utils.py:5


def _to_polar(p: torch.Tensor) -> torch.Tensor:
    """(E,) px, py, pz -> (pt, eta, phi) with the reference's regularisers (hungarian_mse/utils.py:8-28): pt = sqrt(px^2 + py^2 + eps),
    eta = asinh(pz / (pt + eps)), phi = atan2(py + eps, px + eps); the energy of a 4-vector is dropped."""
    if p.shape[-1] not in (3, 4):
        raise ValueError(f"Wrong last dimension of p. Should be 3 or 4 but found: {p.shape[-1]}.")
    xyz = p[..., -3:]
    pt = torch.sqrt(xyz[..., 0] ** 2 + xyz[..., 1] ** 2 + _HEPS)
    return torch.stack((pt, torch.asinh(xyz[..., 2] / (pt + _HEPS)), torch.atan2(xyz[..., 1] + _HEPS, xyz[..., 0] + _HEPS)), dim=-1)


def _relative_polar(p: torch.Tensor, jet: torch.Tensor) -> torch.Tensor:
    """Polar coordinates relative to the jet axis (hungarian_mse/utils.py:35-49): pt / (pt_jet + eps), eta - eta_jet and
    phi - phi_jet wrapped into [-pi, pi).  Written out of place, so that -- unlike the reference, whose in-place updates of
    unbind() views raise under autograd -- the gradient reaches the reconstruction in the relative modes too."""
    import math
    pp, jp = _to_polar(p), _to_polar(jet).unsqueeze(-2)
    dphi = torch.remainder(pp[..., 2] - jp[..., 2] + math.pi, 2 * math.pi) - math.pi
    return torch.stack((pp[..., 0] / (jp[..., 0] + _HEPS), pp[..., 1] - jp[..., 1], dphi), dim=-1)


def _polar_to_cartesian(p: torch.Tensor) -> torch.Tensor:
    """(pt, eta, phi) -> (px, py, pz) as the reference computes it (hungarian_mse/utils.py:52-71).  Its py line reads
    ``pt * torch.cos(phi)`` (:63, a slip for sin); reproduced, because the matching and the loss value depend on it."""
    pt, eta, phi = p[..., -3], p[..., -2], p[..., -1]
    return torch.stack((pt * torch.cos(phi), pt * torch.cos(phi), pt * torch.sinh(eta)), dim=-1)


def hungarian_preprocess(recons: torch.Tensor, target: torch.Tensor, abs_coord: bool = True, polar_coord: bool = False):
    """The four coordinate options of hungarian_mse.py:60-100: absolute Cartesian (identity), absolute polar, and -- relative to
    the TARGET jet's axis -- relative polar or relative Cartesian."""
    for t in (target, recons):
        if t.shape[-1] not in (3, 4):
            raise ValueError(f"Wrong last dimension of p. Should be 3 or 4 but found: {t.shape[-1]}.")
    target = target.to(recons.device)
    if abs_coord:
        return (_to_polar(recons), _to_polar(target)) if polar_coord else (recons, target)
    jet = target.sum(dim=-2)
    r, t = _relative_polar(recons, jet), _relative_polar(target, jet)
    return (r, t) if polar_coord else (_polar_to_cartesian(r), _polar_to_cartesian(t))


class HungarianMSELoss(nn.Module):
    """Permutation-invariant MSE of reference utils/losses/hungarian_mse/hungarian_mse.py (:6-58) with the matching solved on
    the device for the whole batch (`gj_assignment`) instead of `scipy.optimize.linear_sum_assignment` jet by jet on the host
    (:51-52): cost = cdist(recons, target) in the chosen coordinates, recons_shuffle[b] = recons[b, matching[b]],
    loss = MSELoss(recons_shuffle, target).  The gradient reaches `recons` through the coordinate map and the gather."""

    def forward(self, recons: torch.Tensor, target: torch.Tensor, abs_coord: bool = True, polar_coord: bool = False):
        from .anomaly import assignment
        self.abs_coord, self.polar_coord, self.device = abs_coord, polar_coord, recons.device
        recons, target = hungarian_preprocess(recons, target, abs_coord=abs_coord, polar_coord=polar_coord)
        match, _ = assignment(recons, target)
        match = match.to(recons.device)
        recons_shuffle = torch.gather(recons, 1, match.unsqueeze(-1).expand(-1, -1, recons.shape[-1]))
        return nn.functional.mse_loss(recons_shuffle, target)


class _EMD(torch.autograd.Function):
    """Per-jet EMD (float64) of [pt, eta, phi] jets; backward returns the kernel's dEMD/dp, scaled per jet."""

    @staticmethod
    def forward(ctx, p, q, R, beta, norm, periodic_phi):
        from .anomaly import _emd_solve
        e, _, dp, _ = _emd_solve(p, q, R, beta, norm, periodic_phi, want_grad=ctx.needs_input_grad[0])
        ctx.save_for_backward(dp)
        ctx.p_meta = (p.dtype, p.device)
        return e

    @staticmethod
    def backward(ctx, g):
        dp, = ctx.saved_tensors
        dtype, device = ctx.p_meta
        return (dp.double() * g.to(dp.device, torch.float64)[:, None, None]).to(device=device, dtype=dtype), None, None, None, None, None


class EMDLoss(nn.Module):
    """Exact energy mover's distance between reconstructed and target jets (the loss reference utils/losses/emd_loss.py builds
    from jetnet.losses.EMDLoss), solved on the device for the whole batch: ``anomaly.emd`` per jet, reduced by ``reduction``
    ("sum" over jets, as ``ChamferLoss`` sums; "mean"; "none" for the (B,) vector).  recons (B, Np, D) receives the gradient,
    target (B, Nq, D) does not; D = 3 ([pt, eta, phi]) or, with ``polar_coord=False``, Cartesian 3- / 4-vectors converted by the
    differentiable ``_to_polar``.  Particle weights are max(pt, 0): a reconstructed particle with pt <= 0 gets no pt gradient."""

    def __init__(self, R: float = 1.0, beta: float = 1.0, norm: bool = False, periodic_phi: bool = False, polar_coord: bool = True,
                 reduction: str = "sum"):
        super().__init__()
        if reduction not in ("sum", "mean", "none"):
            raise ValueError("reduction must be 'sum', 'mean' or 'none'")
        if not (R > 0 and beta > 0):
            raise ValueError(f"R and beta must be positive, got R={R}, beta={beta}")
        self.R, self.beta, self.norm, self.periodic_phi = float(R), float(beta), bool(norm), bool(periodic_phi)
        self.polar_coord, self.reduction = bool(polar_coord), reduction

    def forward(self, recons: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        from .anomaly import _emd_polar
        if target.requires_grad:
            raise NotImplementedError("the EMD kernel differentiates w.r.t. the reconstruction only")
        p = _emd_polar(recons, self.polar_coord)
        q = _emd_polar(target.to(recons.device), self.polar_coord)
        e = _EMD.apply(p, q, self.R, self.beta, self.norm, self.periodic_phi)
        if self.reduction == "sum":
            e = e.sum()
        elif self.reduction == "mean":
            e = e.mean()
        return e.to(recons.dtype)
