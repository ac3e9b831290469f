"""Anomaly-score distances of reference utils/jet_analysis/anomaly_detection.py (:454-510) on one kernel launch:
``mse``, ``chamfer`` (Euclidean norm) and ``chamfer_lorentz`` with the reference's signatures and return shapes, the
optimal-matching scores ``hungarian`` / ``hungarian_lorentz``, and the exact energy mover's distance ``emd``.

The reference builds the (B, N, N, D) difference tensor and, in the batched form, goes through a DataLoader with one
host <-> device round trip per batch (:471-481); here a CTA per jet keeps the two particle sets in shared memory and
writes the per-particle minima.  There is no CPU fallback: the inputs are moved to the CUDA device.
"""
from __future__ import annotations

import torch

from . import _lib


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("gnn_jet_autoencoder_b200.anomaly needs a CUDA device (there is no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def mse(p: torch.Tensor, q: torch.Tensor, dim: int = -1) -> torch.Tensor:
    """anomaly_detection.py:454-455: squared difference summed over ``dim`` (plain elementwise arithmetic)."""
    return ((p - q) ** 2).sum(dim=dim)


def _pair_min(p: torch.Tensor, q: torch.Tensor, lorentz: bool) -> torch.Tensor:
    if p.dim() != 3 or q.dim() != 3 or p.shape[0] != q.shape[0] or p.shape[2] != q.shape[2]:
        raise ValueError(f"expected (B, N, D) jets with equal B and D, got {tuple(p.shape)} and {tuple(q.shape)}")
    if p.shape[1] != q.shape[1]:
        raise RuntimeError("the reference adds the two per-particle minima elementwise: both jets need the same number of "
                           f"particles (got {p.shape[1]} and {q.shape[1]})")
    if lorentz and p.shape[2] != 4:
        raise ValueError("chamfer_lorentz needs 4-vectors (E, px, py, pz)")
    dev = p.device if p.is_cuda else _device()
    pc = p.detach().to(device=dev, dtype=torch.float32).contiguous()
    qc = q.detach().to(device=dev, dtype=torch.float32).contiguous()
    B, N, D = pc.shape
    out = torch.empty((2, B, N), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().gj_pair_min_dist(B, N, N, D, 1 if lorentz else 0, pc.data_ptr(), qc.data_ptr(), out[0].data_ptr(),
                                                out[1].data_ptr(), torch.cuda.current_stream().cuda_stream), "gj_pair_min_dist")
    return (out[0] + out[1]).to(p.dtype if p.dtype.is_floating_point else torch.float32)


def _batched(fn, p, q, batch_size):
    """anomaly_detection.py:471-481: with a positive ``batch_size`` the reference walks the data in batches on DEVICE and
    returns a CPU tensor; otherwise the result stays on the inputs' device."""
    if batch_size is not None and batch_size > 0:
        return torch.cat([fn(p[i:i + batch_size], q[i:i + batch_size]).cpu() for i in range(0, p.shape[0], batch_size)], dim=0)
    out = fn(p, q)
    return out if p.is_cuda else out.cpu()


def chamfer(p: torch.Tensor, q: torch.Tensor, batch_size: int = -1) -> torch.Tensor:
    """anomaly_detection.py:459-488: (B, N) tensor  min_j |p_i - q_j|_2 + min_i' |p_i' - q_i|_2  (per-particle sums of the two
    nearest-neighbour distances; L2 norm, not squared)."""
    return _batched(lambda a, b: _pair_min(a, b, False), p, q, batch_size)


def chamfer_lorentz(p: torch.Tensor, q: torch.Tensor, batch_size: int = -1) -> torch.Tensor:
    """anomaly_detection.py:491-510: the same with the Lorentz norm squared E^2 - px^2 - py^2 - pz^2 of the differences."""
    return _batched(lambda a, b: _pair_min(a, b, True), p, q, batch_size)


def assignment(p: torch.Tensor, q: torch.Tensor, lorentz: bool = False):
    """Optimal particle matching per jet on the device: (col_for_row (B, N) int64, total_cost (B,)) with
    col_for_row[b] == scipy.optimize.linear_sum_assignment(cost[b])[1] for cost = cdist(p, q) (or the Lorentz norm squared of
    the differences) -- the matching step of anomaly_detection.py:537-541 / :579-585 and hungarian_mse.py:51-52."""
    if p.dim() != 3 or p.shape != q.shape:
        raise ValueError(f"expected two (B, N, D) tensors of equal shape, got {tuple(p.shape)} and {tuple(q.shape)}")
    if lorentz and p.shape[2] != 4:
        raise ValueError("the Lorentz norm needs 4-vectors (E, px, py, pz)")
    dev = p.device if p.is_cuda else _device()
    pc = p.detach().to(device=dev, dtype=torch.float32).contiguous()
    qc = q.detach().to(device=dev, dtype=torch.float32).contiguous()
    B, N, D = pc.shape
    match = torch.empty((B, N), device=dev, dtype=torch.int32)
    total = torch.empty((B,), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().gj_assignment(B, N, D, 1 if lorentz else 0, pc.data_ptr(), qc.data_ptr(), match.data_ptr(),
                                             total.data_ptr(), torch.cuda.current_stream().cuda_stream), "gj_assignment")
    return match.long(), total


def _hungarian(p: torch.Tensor, q: torch.Tensor, lorentz: bool) -> torch.Tensor:
    match, _ = assignment(p, q, lorentz)
    pd = p.to(match.device)
    # anomaly_detection.py:543-546: p_shuffle[b] = p[b, matching[b]], then the particle-wise squared error against q
    p_shuffle = torch.gather(pd, 1, match.unsqueeze(-1).expand(-1, -1, pd.shape[-1]))
    return mse(p_shuffle, q.to(match.device))


def hungarian(p: torch.Tensor, q: torch.Tensor, batch_size: int = -1) -> torch.Tensor:
    """anomaly_detection.py:513-547: (B, N) squared errors after the optimal (Euclidean-cost) matching of the particles."""
    return _batched(lambda a, b: _hungarian(a, b, False), p, q, batch_size)


def hungarian_lorentz(p: torch.Tensor, q: torch.Tensor, batch_size: int = -1) -> torch.Tensor:
    """anomaly_detection.py:550-590: the same with the Lorentz norm squared of the differences as the matching cost."""
    return _batched(lambda a, b: _hungarian(a, b, True), p, q, batch_size)


def _emd_polar(x: torch.Tensor, polar_coord: bool) -> torch.Tensor:
    """[pt, eta, phi] jets as ``gj_emd`` takes them: as given, or converted from Cartesian 3- / 4-vectors like
    ``losses.hungarian_preprocess`` does."""
    from .losses import _to_polar
    if x.dim() != 3:
        raise ValueError(f"expected (B, N, D) jets, got {tuple(x.shape)}")
    if polar_coord:
        if x.shape[-1] != 3:
            raise ValueError(f"polar_coord=True expects [pt, eta, phi] jets (B, N, 3), got {tuple(x.shape)}")
        return x
    return _to_polar(x)


def _emd_solve(p: torch.Tensor, q: torch.Tensor, R: float, beta: float, norm: bool, periodic_phi: bool, want_flow: bool = False,
               want_grad: bool = False, want_potentials: bool = False, first: int = 0):
    """One ``gj_emd`` launch on [pt, eta, phi] jets p (B, Np, 3), q (B, Nq, 3): (emd (B,) float64, flow (B, Np, Nq) float64,
    dEMD/dp (B, Np, 3) float32, potentials (B, Np+1+Nq+1) float64), the last three None unless asked for.  Raises ``ValueError``
    naming the jets (numbered from ``first``) with a non-finite pt, eta or phi (the solver does not run on them), and ``RuntimeError`` if a jet's solver did
    not converge."""
    if p.dim() != 3 or q.dim() != 3 or p.shape[0] != q.shape[0] or p.shape[2] != 3 or q.shape[2] != 3:
        raise ValueError(f"expected (B, Np, 3) and (B, Nq, 3) jets, got {tuple(p.shape)} and {tuple(q.shape)}")
    dev = p.device if p.is_cuda else _device()
    pc = p.detach().to(device=dev, dtype=torch.float32).contiguous()
    qc = q.detach().to(device=dev, dtype=torch.float32).contiguous()
    B, Np, Nq = pc.shape[0], pc.shape[1], qc.shape[1]
    f64 = dict(device=dev, dtype=torch.float64)
    emd = torch.empty((B,), **f64)
    flow = torch.empty((B, Np, Nq), **f64) if want_flow else None
    dp = torch.empty((B, Np, 3), device=dev, dtype=torch.float32) if want_grad else None
    pot = torch.empty((B, Np + Nq + 2), **f64) if want_potentials else None
    status = torch.empty((B,), device=dev, dtype=torch.int32)
    flags = (_lib.GJ_EMD_NORM if norm else 0) | (_lib.GJ_EMD_PERIODIC_PHI if periodic_phi else 0)
    ptr = lambda t: t.data_ptr() if t is not None else None
    with torch.cuda.device(dev):
        _lib.check(_lib.load().gj_emd(B, Np, Nq, pc.data_ptr(), qc.data_ptr(), float(R), float(beta), flags, emd.data_ptr(), ptr(flow),
                                      ptr(dp), ptr(pot), status.data_ptr(), None, 0, torch.cuda.current_stream().cuda_stream), "gj_emd")
    nonfinite = [first + k for k in (status == 2).nonzero().flatten().tolist()]
    if nonfinite:
        raise ValueError(f"gj_emd: jet(s) {nonfinite} have a NaN or infinite pt, eta or phi: their EMD is not defined")
    bad = int((status != 0).sum())
    if bad:
        raise RuntimeError(f"gj_emd: the transport solver did not converge for {bad} of {B} jets")
    return emd, flow, dp, pot


def emd(p: torch.Tensor, q: torch.Tensor, R: float = 1.0, beta: float = 1.0, norm: bool = False, periodic_phi: bool = False,
        polar_coord: bool = True, batch_size: int = -1, return_flow: bool = False):
    """Exact energy mover's distance per jet (energyflow.emd.emd's definition; the EMD score of anomaly_detection.py), solved for
    the whole batch in one launch: (B,) float64 tensor of

        EMD = min_f sum_ij f_ij (theta_ij / R)^beta + |W_p - W_q|,  sum_j f_ij <= w_i, sum_i f_ij <= w'_j, sum f = min(W_p, W_q)

    with weights w = max(pt, 0) and theta_ij = sqrt(deta^2 + dphi^2) (dphi wrapped into [-pi, pi) with ``periodic_phi``).
    p (B, Np, 3) and q (B, Nq, 3) are [pt, eta, phi] jets, or Cartesian 3- / 4-vectors with ``polar_coord=False``; Np and Nq
    may differ (at most 150 each).  ``norm`` divides each jet's weights by its total.  ``return_flow`` also returns the optimal
    flow (B, Np, Nq) float64.  A positive ``batch_size`` walks the jets in batches and returns CPU tensors, like the other
    scores here.  Raises ``ValueError`` naming the jets with a NaN or infinite pt, eta or phi (their EMD is not defined), and
    ``RuntimeError`` if a jet's solver did not converge."""
    def one(a, b, first=0):
        dev = a.device if a.is_cuda else _device()
        e, f, _, _ = _emd_solve(_emd_polar(a.to(dev), polar_coord), _emd_polar(b.to(dev), polar_coord), R, beta, norm, periodic_phi,
                                want_flow=return_flow, first=first)
        return e, f
    if batch_size is not None and batch_size > 0 and p.shape[0] > 0:
        parts = [one(p[i:i + batch_size], q[i:i + batch_size], i) for i in range(0, p.shape[0], batch_size)]
        e = torch.cat([x[0].cpu() for x in parts])
        f = torch.cat([x[1].cpu() for x in parts]) if return_flow else None
    else:
        e, f = one(p, q)
        if not p.is_cuda:
            e, f = e.cpu(), (f.cpu() if return_flow else None)
    return (e, f) if return_flow else e
