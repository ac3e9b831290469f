"""Float64 reference of the energy mover's distance (energyflow.emd.emd's definition, Komiske, Metodiev, Thaler, PRL 123,
041801) for the tests of ``gj_emd``: one linear program per jet through ``scipy.optimize.linprog(method="highs")``, and a
checker that certifies a (flow, potentials) pair returned by the kernel as optimal.

Jets are (N, 3) arrays [pt, eta, phi]; weights w = max(pt, 0); theta_ij = sqrt(deta^2 + dphi^2) (dphi wrapped into [-pi, pi)
with periodic_phi); cost (theta / R)^beta;
    EMD = min_f sum_ij f_ij c_ij + |W_p - W_q|,  sum_j f_ij <= w_i, sum_i f_ij <= w'_j, sum_ij f_ij = min(W_p, W_q).
norm divides each non-empty jet's weights by its total (the imbalance term is then 0, or 1 against an empty jet).
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import linprog


def weights_and_cost(p, q, R=1.0, beta=1.0, norm=False, periodic_phi=False):
    """(a (Np,), b (Nq,), C (Np, Nq), total of a, total of b) in float64; the totals are exactly 0 or 1 with ``norm``."""
    p, q = np.asarray(p, np.float64), np.asarray(q, np.float64)
    a, b = np.maximum(p[:, 0], 0.0), np.maximum(q[:, 0], 0.0)
    sa, sb = a.sum(), b.sum()
    if norm:
        a = a / sa if sa > 0 else a
        b = b / sb if sb > 0 else b
        sa, sb = float(sa > 0), float(sb > 0)
    de = p[:, None, 1] - q[None, :, 1]
    dphi = p[:, None, 2] - q[None, :, 2]
    if periodic_phi:
        dphi = np.mod(dphi + np.pi, 2 * np.pi) - np.pi
    C = (np.sqrt(de * de + dphi * dphi) / R) ** beta
    return a, b, C, sa, sb


def emd_lp(p, q, R=1.0, beta=1.0, norm=False, periodic_phi=False):
    """(emd, flow (Np, Nq), duals) of one jet pair; duals = (row marginals (Np,), column marginals (Nq,), total-flow marginal)
    of linprog's inequality and equality constraints (zeros when no flow can move)."""
    a, b, C, sa, sb = weights_and_cost(p, q, R, beta, norm, periodic_phi)
    n, m = C.shape
    imbalance = abs(sa - sb)
    total = min(a.sum(), b.sum())
    if total <= 0:
        return imbalance, np.zeros((n, m)), (np.zeros(n), np.zeros(m), 0.0)
    A_ub = np.zeros((n + m, n * m))
    for i in range(n):
        A_ub[i, i * m:(i + 1) * m] = 1.0
    for j in range(m):
        A_ub[n + j, j::m] = 1.0
    res = linprog(C.ravel(), A_ub=A_ub, b_ub=np.concatenate([a, b]), A_eq=np.ones((1, n * m)), b_eq=[total], bounds=(0, None),
                  method="highs")
    assert res.status == 0, res.message
    duals = (res.ineqlin.marginals[:n], res.ineqlin.marginals[n:], float(res.eqlin.marginals[0]))
    return float(res.fun) + imbalance, res.x.reshape(n, m), duals


def certify(p, q, flow, potentials, emd_value, R=1.0, beta=1.0, norm=False, periodic_phi=False):
    """Optimality certificate of a kernel result for one jet pair, in the balanced form the kernel solves (a dummy row of weight
    max(W_q - W_p, 0) and a dummy column of weight max(W_p - W_q, 0), at cost 1 to every particle and 0 to each other).
    flow (Np, Nq): transport between the particles (the dummies take the rest); potentials (Np + 1 + Nq + 1): u_0..u_Np,
    v_0..v_Nq.  Returns the worst violations, each relative to the problem's scale:
      primal: negative flow, row / column sums above the weights, total flow off min(W_p, W_q);
      dual:   u_i + v_j above c_ij on any arc (dummy arcs included);
      gap:    |primal objective - dual objective| and |primal objective - emd_value|."""
    a, b, C, sa, sb = weights_and_cost(p, q, R, beta, norm, periodic_phi)
    n, m = C.shape
    flow, pot = np.asarray(flow, np.float64), np.asarray(potentials, np.float64)
    u, ud, v, vd = pot[:n], pot[n], pot[n + 1:n + 1 + m], pot[n + 1 + m]
    scale = max(a.sum(), b.sum(), 1e-300)
    rows, cols = flow.sum(1), flow.sum(0)
    primal = max(float(-flow.min(initial=0.0)), float((rows - a).max(initial=0.0)), float((cols - b).max(initial=0.0)),
                 abs(float(flow.sum()) - min(a.sum(), b.sum()))) / scale
    cmax = max(float(C.max(initial=0.0)), 1.0)
    dual = max(float((u[:, None] + v[None, :] - C).max(initial=-np.inf)), float((u + vd - 1.0).max(initial=-np.inf)),
               float((ud + v - 1.0).max(initial=-np.inf)), ud + vd, 0.0) / cmax
    dr, dc = max(sb - sa, 0.0), max(sa - sb, 0.0)
    obj_p = float((flow * C).sum() + (a - rows).sum() + (b - cols).sum())
    obj_d = float(a @ u + b @ v + dr * ud + dc * vd)
    den = max(abs(obj_p), 1e-12)
    return {"primal": primal, "dual": dual, "gap": abs(obj_p - obj_d) / den, "value": abs(obj_p - float(emd_value)) / den}
