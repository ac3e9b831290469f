/*
 * gnnjet_b200.h -- C-ABI of the B200-native GraphNet message-passing path.
 *
 * The reference (zichunhao/gnn-jet-autoencoder) is pure Python/PyTorch and has no FFI; the
 * boundary it exposes for this path is the nn.Module surface of models/ (SURVEY.md 8.b).
 * This header is what a binding for that path binds: every entry point is extern "C", takes
 * raw DEVICE pointers + explicit sizes + a cudaStream_t (as void*), returns an int status
 * (0 = ok), allocates nothing the caller must free and keeps no global mutable state apart
 * from a thread-local last-error string.  No torch types appear in any signature.
 *
 * Reference interfaces replaced (paths relative to the reference checkout):
 *   gj_mp_step_fwd / gj_mp_step_bwd  : one iteration of the loop in models/graphnet.py:154-168
 *                                      (_getA :186-223, _edge_conv :273-289, _concat :225-247,
 *                                      _aggregate :249-271) and its autograd adjoint
 *   gj_chamfer_fwd_bwd               : utils/losses/chamfer_loss/chamfer_loss.py:11-42 with
 *                                      utils/losses/chamfer_loss/distance_sq.py:4-77
 *   gj_adam_step_flat                : torch.optim.Adam as built in utils/initialize.py:152-153,
 *                                      with the L1/L2 regulariser gradients of utils/train.py:376-384
 *   gj_optimizer_step_flat           : torch.optim.RMSprop / Adagrad / SGD as built in utils/initialize.py:154-170
 *   gj_latent_mean_fwd/bwd           : models/encoder.py:147-149 ('mean' latent map)
 *   gj_latent_extreme_fwd/bwd        : models/encoder.py:150-155 ('max' / 'min' latent maps)
 *   gj_output_transform_fwd/bwd      : models/decoder.py:123-124 (tanh) and utils/train.py:55-65 (polar clamp)
 *   gj_mse_fwd_bwd                   : utils/train.py:359-361 (nn.MSELoss branch of get_loss)
 *   gj_emd_loss                      : the emd branch of get_loss (utils/train.py:330-385) on utils/losses/emd_loss.py
 *   gj_hungarian_mse_loss            : utils/losses/hungarian_mse/hungarian_mse.py:27-58 as a training loss
 *
 * Tensor layouts: all tensors are dense row-major float32 in HBM.
 *   node features  h      (B, N, H)
 *   packed params  params per message-passing step t, in state_dict order:
 *       edge_net.t.0.weight (E0, 2H+1) | edge_net.t.0.bias (E0) | edge_net.t.1.weight (E1,E0) | ...
 *       node_net.t.0.weight (O0, E_last+H) | node_net.t.0.bias (O0) | node_net.t.1.weight ...
 *     weights are (out, in) row-major exactly as torch.nn.Linear stores them; the first edge
 *     layer's input axis is ordered [h_i (H) | h_j (H) | d_ij (1)] (graphnet.py:220) and the first
 *     node layer's input axis is [sum_j edge (E_last) | h (H)] (graphnet.py:246).
 */
#ifndef GNNJET_B200_H
#define GNNJET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GJ_MAX_LAYERS 8

/* status codes */
#define GJ_OK 0
#define GJ_ERR_INVALID 1     /* bad argument / unsupported shape */
#define GJ_ERR_SMEM 2        /* configuration does not fit the 227 KB shared-memory budget */
#define GJ_ERR_CUDA 3        /* a CUDA runtime call failed; see gj_last_error() */
#define GJ_ERR_WORKSPACE 4   /* workspace too small */

/* precision modes */
#define GJ_PREC_FP32 0       /* SIMT FFMA, fp32 everywhere: <=1e-5 relative vs the fp64 reference */
#define GJ_PREC_BF16 1       /* edge-MLP hidden layers on tcgen05 (bf16 operands, fp32 TMEM accumulators) */

/* distance metric of graphnet.py:314-327 */
#define GJ_METRIC_EUCLIDEAN 0
#define GJ_METRIC_MINKOWSKIAN 1  /* applied only where the current node width is 4 (graphnet.py:155) */

/* One message-passing step (one iteration of graphnet.py:154-168). */
typedef struct gj_mp_desc {
  int32_t batch;                         /* B jets */
  int32_t num_nodes;                     /* N particles per jet */
  int32_t node_in;                       /* H  : width of h entering the step */
  int32_t n_edge_layers;                 /* number of Linear layers in edge_net[t] (>=1) */
  int32_t edge_widths[GJ_MAX_LAYERS];    /* output width of each edge layer */
  int32_t n_node_layers;                 /* number of Linear layers in node_net[t] (>=1) */
  int32_t node_widths[GJ_MAX_LAYERS];    /* output width of each node layer; last one is the step's output width */
  float alpha;                           /* LeakyReLU negative slope (>= 0) used after EVERY layer */
  int32_t metric;                        /* GJ_METRIC_* */
  int32_t precision;                     /* GJ_PREC_* */
  int32_t h_ld;                          /* row stride of h (and dh) in floats; 0 = node_in */
  int32_t h_cols;                        /* columns of each h row that exist in memory (<= h_ld); columns
                                            [h_cols, node_in) are zeros (the F.pad of graphnet.py:152), and with
                                            h_cols = node_in < h_ld the row is cropped (negative pad); 0 = node_in */
} gj_mp_desc;

/* Number of floats in the packed parameter block of one step (0 on invalid desc). */
size_t gj_mp_param_count(const gj_mp_desc* d);

/* Process-wide switch (returns the previous value; set it before the calls it should affect, not inside a CUDA-graph capture that
 * was made with the other value).  In the GJ_PREC_BF16 mode forward results and all data gradients are always bitwise
 * reproducible; PARAMETER gradients are reproducible to fp32 summation order only, because the tile groups of a CTA accumulate
 * into shared tensor-memory accumulators in a timing-dependent order.  on != 0 runs the backward edge kernels with one tile group
 * per CTA: parameter gradients become bitwise reproducible from run to run at roughly 2.5x the backward edge time
 * (the analogue of torch.use_deterministic_algorithms for this path).  GJ_PREC_FP32 is always bitwise reproducible. */
int32_t gj_set_deterministic(int32_t on);

/* Workspace bytes needed by gj_mp_step_fwd (the per-node projections P|Q of the factorised first edge layer). */
size_t gj_mp_step_fwd_workspace(const gj_mp_desc* d);

/* Forward of one step.  h (B,N,h_ld) -> h_out (B,N,node_widths[last]).
 * e_out (required) receives the edge aggregate sum_j EdgeNet(A_ij) (B,N,edge_widths[last]), which
 * gj_mp_step_bwd needs (it is the only tensor saved for backward besides h).
 * Launch sequence: node projections -> fused edge kernel (pair tiles in shared memory / TMEM only) -> node MLP. */
int gj_mp_step_fwd(const gj_mp_desc* d, const float* h, const float* params,
                   float* h_out, float* e_out, void* workspace, size_t workspace_bytes, void* stream);

/* Optional reuse of forward by-products in backward.  gj_mp_step_saved_bytes(d) > 0 means the step runs the fused
 * tensor-core kernels and gj_mp_step_fwd_saving can leave its per-node projections P|Q, the packed bf16 edge parameters
 * and the pair distances d_ij in a caller-owned buffer `saved` of that many bytes (256-byte aligned); passing the same
 * buffer, unmodified, to gj_mp_step_bwd_saved (same desc, h, params) skips their recomputation.  Results are identical to
 * gj_mp_step_fwd / gj_mp_step_bwd.  Both return GJ_ERR_INVALID where gj_mp_step_saved_bytes is 0. */
size_t gj_mp_step_saved_bytes(const gj_mp_desc* d);
/* Number of kernels one gj_mp_step_fwd (backward = 0) or gj_mp_step_bwd / _bwd_saved (backward = 1, with_saved = 0 / 1)
 * call launches for this descriptor (memsets not counted); 0 for an invalid descriptor.  bench.py's gpu_launches adds these up. */
int gj_mp_step_launches(const gj_mp_desc* d, int backward, int with_saved);
int gj_mp_step_fwd_saving(const gj_mp_desc* d, const float* h, const float* params,
                          float* h_out, float* e_out, void* saved, void* workspace, size_t workspace_bytes, void* stream);
int gj_mp_step_bwd_saved(const gj_mp_desc* d, const float* h, const float* e, const float* params,
                         const float* dh_out, float* dh, float* dparams, const void* saved,
                         void* workspace, size_t workspace_bytes, void* stream);

/* A chain of steps (a GraphNet, or encoder + decoder of a training step: the loop of graphnet.py:154-168 and its adjoint)
 * with per-chain instead of per-step helper launches.  Two pieces of every step depend on the parameters only or are needed
 * only at the end of the backward pass: the packed bf16 image of the edge-network weights (one small launch per step) and the
 * fixed-order reduction of the per-CTA parameter-gradient partials (another).  For steps with gj_mp_step_partials_bytes(d) > 0
 * (the fused tensor-core kernels, gj_mp_step_saved_bytes(d) > 0 as well):
 *   gj_mp_steps_pack       : ONE launch writes the parameter images of all n steps into their `saved` buffers (any time after
 *                            the parameters were last updated, before the first gj_mp_step_fwd_packed);
 *   gj_mp_step_fwd_packed  : gj_mp_step_fwd_saving without the packing launch (the image in `saved` is used as it is);
 *   gj_mp_step_bwd_deferred: gj_mp_step_bwd_saved without the reduction: the per-CTA partials are left in the caller-owned
 *                            buffer `partials` (gj_mp_step_partials_bytes(d) bytes, 256-byte aligned) and no dparams is written;
 *   gj_mp_steps_reduce     : ONE launch reduces the partials of all n steps into their dparams blocks (same summation order as
 *                            gj_mp_step_bwd_saved: the results are identical).
 * Every function returns GJ_ERR_INVALID for a step with gj_mp_step_partials_bytes(d) == 0; n <= 64. */
size_t gj_mp_step_partials_bytes(const gj_mp_desc* d);
int gj_mp_steps_pack(int32_t n, const gj_mp_desc* const* descs, const float* const* params, void* const* saved, void* stream);
int gj_mp_step_fwd_packed(const gj_mp_desc* d, const float* h, const float* params,
                          float* h_out, float* e_out, void* saved, void* workspace, size_t workspace_bytes, void* stream);
int gj_mp_step_bwd_deferred(const gj_mp_desc* d, const float* h, const float* e, const float* params,
                            const float* dh_out, float* dh, const void* saved, void* partials,
                            void* workspace, size_t workspace_bytes, void* stream);
int gj_mp_steps_reduce(int32_t n, const gj_mp_desc* const* descs, const void* const* partials, float* const* dparams, void* stream);

/* Workspace bytes needed by gj_mp_step_bwd (P|Q, their gradients, de, per-CTA parameter-gradient partials). */
size_t gj_mp_step_bwd_workspace(const gj_mp_desc* d);

/* Backward of one step: recomputes the edge MLP per tile (nothing N^2-sized is ever stored).
 * in : h, e (saved by forward), params, dh_out (B,N,out)
 * out: dh (B,N,h_ld; the first h_cols columns of every row are OVERWRITTEN, others untouched),
 *      dparams (packed like params; OVERWRITTEN with the batch-summed gradient, deterministic reduction order). */
int gj_mp_step_bwd(const gj_mp_desc* d, const float* h, const float* e, const float* params,
                   const float* dh_out, float* dh, float* dparams,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Chamfer terms and gradient w.r.t. p (the reconstruction).
 * p (B,Np,D), q (B,Nq,D), D in {3,4}; norm: 0 cartesian, 1 minkowskian/polar (2*p0^2 - sum p^2).  For D == 3 the
 * PAIRWISE distances are always cartesian (distance_sq.py:43-44) while the jet term keeps the requested norm
 * (chamfer_loss.py:40 calls normsq directly: p0^2 - p1^2 - p2^2).
 * terms[0] = sum_b [sum_i min_j dist + sum_j min_i dist]   terms[1] = sum_b normsq(sum p - sum q)
 * terms[2] = w_chamfer * terms[0] + w_jet * terms[1]
 * (overwritten; deterministic: per-jet partials are written to jet_terms (B,2), which is also an
 * output, and reduced by a single block in a fixed order).
 * dp (B,Np,D), may be NULL: gradient of terms[2] w.r.t. p (through the arg-mins, first index on ties).
 * The loss chamfer_loss.py:35-41 builds is (w_chamfer, w_jet) = (1, jet_features_weight); the value it
 * RETURNS (:42) is (0, 1). */
int gj_chamfer_fwd_bwd(int32_t batch, int32_t np_, int32_t nq, int32_t dim, int32_t norm,
                       float w_chamfer, float w_jet, const float* p, const float* q,
                       float* jet_terms, float* terms, float* dp, void* stream);

/* Per-particle nearest-neighbour distances of the anomaly scores (utils/jet_analysis/anomaly_detection.py: chamfer
 * :459-488, chamfer_lorentz :491-510).  p (B,Np,D), q (B,Nq,D), D <= 4.
 * lorentz == 0: min_pq[b][i] = min_j |p_i - q_j|_2, min_qp[b][j] = min_i |p_i - q_j|_2;
 * lorentz == 1 (D == 4): the same minima of E^2 - px^2 - py^2 - pz^2 of the difference (no square root, may be negative).
 * The reference's score is min_pq + min_qp (elementwise, Np == Nq). */
int gj_pair_min_dist(int32_t batch, int32_t np_, int32_t nq, int32_t dim, int32_t lorentz, const float* p, const float* q,
                     float* min_pq, float* min_qp, void* stream);

/* Optimal assignment (minimum total cost perfect matching) between the N particles of p and of q, per jet: the matching of
 * utils/jet_analysis/anomaly_detection.py hungarian :513-547 / hungarian_lorentz :550-590 and of
 * utils/losses/hungarian_mse/hungarian_mse.py:51-56, which call scipy.optimize.linear_sum_assignment jet by jet on the host.
 * cost(i, j) = |p_i - q_j|_2 (lorentz == 0) or E^2 - px^2 - py^2 - pz^2 of p_i - q_j (lorentz == 1, D == 4).
 * col_for_row (B,N) int32: column (particle of q) assigned to row i (particle of p) -- linear_sum_assignment(cost)[1];
 * total_cost (B), may be NULL: the assignment's cost.  N <= 220 (the cost matrix lives in shared memory). */
int gj_assignment(int32_t batch, int32_t n, int32_t dim, int32_t lorentz, const float* p, const float* q,
                  int32_t* col_for_row, float* total_cost, void* stream);

/* Exact energy mover's distance per jet, as energyflow.emd.emd defines it (Komiske, Metodiev, Thaler, PRL 123, 041801): the
 * EMD scores of utils/jet_analysis/anomaly_detection.py (through energyflow) and the loss of utils/losses/emd_loss.py (through
 * jetnet.losses.EMDLoss), both computed jet by jet on the host there.
 * p (B,Np,3), q (B,Nq,3) as [pt, eta, phi]; weights w = max(pt, 0); theta_ij = sqrt(deta^2 + dphi^2) (dphi wrapped into
 * [-pi, pi) with GJ_EMD_PERIODIC_PHI);
 *   EMD = min_{f >= 0} sum_ij f_ij (theta_ij / R)^beta + |W_p - W_q|,
 *         sum_j f_ij <= w_i, sum_i f_ij <= w'_j, sum_ij f_ij = min(W_p, W_q)        (W: total weight of a jet).
 * GJ_EMD_NORM divides each non-empty jet's weights by its total (no imbalance term; an empty jet against a non-empty one gives 1).
 * The problem is solved exactly as a balanced transportation problem with a dummy row (index Np, weight max(W_q - W_p, 0)) and a
 * dummy column (index Nq, weight max(W_p - W_q, 0)) at cost 1 to every particle and 0 to each other; one CTA per jet, successive
 * shortest paths with fp64 potentials and flows.  1 <= Np, Nq <= 150, R > 0, beta > 0.
 * emd_out (B) fp64.  Optional (NULL = not written):
 *   flow_out (B,Np,Nq) fp64: the optimal flow between the real particles (with GJ_EMD_NORM in normalised units);
 *   dp_out (B,Np,3) fp32: gradient of emd_out w.r.t. p -- d/d(eta, phi) = sum_j f_ij beta theta_ij^(beta-2) / R^beta (deta, dphi)
 *     (0 at theta = 0); d/dpt = the row's dual minus the dual of the dummy that absorbs the change (chain rule of the
 *     normalisation with GJ_EMD_NORM), 0 where pt <= 0;
 *   potentials_out (B, Np+1+Nq+1) fp64: optimal duals (u_0..u_Np, v_0..v_Nq) of the balanced problem, u_i + v_j <= c_ij with
 *     equality where flow moves, and sum_i a_i u_i + sum_j b_j v_j = EMD;
 *   status_out (B) int32: 0 converged, 1 augmentation cap N1 N2 + 4 (N1 + N2) + 64 reached, N1 = Np + 1, N2 = Nq + 1
 *     (emd_out is then not optimal).
 * gj_emd_workspace returns 0 for every shape (the solver's state lives in shared memory): workspace may be NULL. */
#define GJ_EMD_NORM 1
#define GJ_EMD_PERIODIC_PHI 2
size_t gj_emd_workspace(int32_t batch, int32_t np_, int32_t nq);
int gj_emd(int32_t batch, int32_t np_, int32_t nq, const float* p, const float* q, float R, float beta, int32_t flags,
           double* emd_out, double* flow_out, float* dp_out, double* potentials_out, int32_t* status_out,
           void* workspace, size_t workspace_bytes, void* stream);

/* The EMD as a training loss (the `emd` branch of get_loss, utils/train.py:330-385, on utils/losses/emd_loss.py): gj_emd's solver,
 * one CTA per jet, on the training step's layout, with the gradient scaled and in the input's own coordinates.
 * p (B,N,D) is the reconstruction, q (B,N,D) the target, fp32, D in {3,4}:
 *   GJ_EMD_COORDS_POLAR     : D == 3, [pt, eta, phi], as gj_emd takes them;
 *   GJ_EMD_COORDS_CARTESIAN : (px, py, pz) or (E, px, py, pz), converted on load as losses._to_polar does
 *                             (pt = sqrt(px^2 + py^2 + 1e-16), eta = asinh(pz / (pt + 1e-16)), phi = atan2(py + 1e-16, px + 1e-16));
 *                             E does not enter the EMD.
 * R, beta, flags (GJ_EMD_NORM, GJ_EMD_PERIODIC_PHI) as for gj_emd; 1 <= N <= 150.
 * terms (3) fp32, overwritten: terms[0] = sum_b EMD_b, terms[1] = 0, terms[2] = scale * terms[0] (the slots of gj_chamfer_fwd_bwd);
 *   the per-jet EMDs are fp64 in the workspace and summed in a fixed order (bitwise reproducible).
 * failed (1) fp32, overwritten: number of jets whose solver stopped at the augmentation cap (their EMD and gradient are not optimal).
 * dp (B,N,D) fp32, may be NULL: scale * dEMD_b/dp as gj_emd's dp_out (rounded to fp32 first), through the Jacobian of the
 *   conversion in Cartesian coordinates; the E component is 0.
 * Two launches (the solver, then the sum), no host synchronisation, capturable in a CUDA graph.  Every argument is checked on the
 * host before any launch; workspace_bytes >= gj_emd_loss_workspace(B, N). */
#define GJ_EMD_COORDS_POLAR 0
#define GJ_EMD_COORDS_CARTESIAN 1
size_t gj_emd_loss_workspace(int32_t batch, int32_t n);
int gj_emd_loss(int32_t batch, int32_t n, int32_t dim, int32_t coords, const float* p, const float* q, float R, float beta,
                int32_t flags, float scale, float* terms, float* failed, float* dp, void* workspace, size_t workspace_bytes,
                void* stream);

/* The Hungarian-matched MSE as a training loss (utils/losses/hungarian_mse/hungarian_mse.py:27-58, losses.HungarianMSELoss): per jet
 * the coordinate map T of `coords`, the optimal matching of gj_assignment on cost |T(p)_i - T(q)_j|_2, and the squared error of the
 * reconstruction gathered with the matching, one CTA per jet.  p (B,N,D) is the reconstruction, q (B,N,D) the target, fp32, D in {3,4};
 * T (losses.hungarian_preprocess, the last three components of p / q taken as (px, py, pz)):
 *   GJ_HMSE_ABS_CARTESIAN : identity, D' = D;
 *   GJ_HMSE_ABS_POLAR     : (pt, eta, phi) as losses._to_polar (pt = sqrt(px^2 + py^2 + 1e-16), eta = asinh(pz / (pt + 1e-16)),
 *                           phi = atan2(py + 1e-16, px + 1e-16)), D' = 3;
 *   GJ_HMSE_REL_POLAR     : relative to the axis of the TARGET jet (the sum of q's particles, converted the same way):
 *                           (pt / (pt_jet + 1e-16), eta - eta_jet, phi - phi_jet wrapped into [-pi, pi)), D' = 3;
 *   GJ_HMSE_REL_CARTESIAN : those relative coordinates as (pt cos phi, pt cos phi, pt sinh eta) (the reference's py), D' = 3.
 * With sigma = col_for_row of the matching, the loss of jet b is L_b = sum_i |T(p)_sigma(i) - T(q)_i|^2 (fp64 in the workspace).
 * terms (3) fp32, overwritten: terms[0] = sum_b L_b, terms[1] = 0, terms[2] = scale * terms[0] (the slots of gj_chamfer_fwd_bwd;
 *   summed in a fixed order, bitwise reproducible).  HungarianMSELoss's mean is scale = 1 / (B N D').
 * dp (B,N,D) fp32, overwritten: d terms[2] / dp = 2 scale (T(p)_k - T(q)_sigma^-1(k)) J_T(p_k) in p's own coordinates; no gradient
 *   flows through the matching or the target's axis, and the E component of a 4-vector is 0 except with GJ_HMSE_ABS_CARTESIAN.
 * col_for_row (B,N) int32, may be NULL: the matching, as gj_assignment returns it for T(p), T(q).
 * 1 <= N <= 220.  Two launches (the matching and loss, then the sum), no host synchronisation, capturable in a CUDA graph.  Every
 * argument is checked on the host before any launch; workspace_bytes >= gj_hungarian_mse_loss_workspace(B, N). */
#define GJ_HMSE_ABS_CARTESIAN 0
#define GJ_HMSE_ABS_POLAR 1
#define GJ_HMSE_REL_POLAR 2
#define GJ_HMSE_REL_CARTESIAN 3
size_t gj_hungarian_mse_loss_workspace(int32_t batch, int32_t n);
int gj_hungarian_mse_loss(int32_t batch, int32_t n, int32_t dim, int32_t coords, const float* p, const float* q, float scale,
                          float* terms, float* dp, int32_t* col_for_row, void* workspace, size_t workspace_bytes, void* stream);

/* Flat fused Adam (torch.optim.Adam defaults: no weight decay, no amsgrad) over n floats.
 * grad_scale multiplies the incoming gradient, l1_lambda*sign(p) and 2*l2_lambda*p are added to it
 * (utils/train.py:376-384).  step is the 1-based step count of this update. */
int gj_adam_step_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n,
                      float lr, float beta1, float beta2, float eps, int32_t step,
                      float grad_scale, float l1_lambda, float l2_lambda, void* stream);

/* The other optimisers utils/initialize.py:154-170 can select, over the same flat buffers and with the same regulariser terms:
 * GJ_OPT_RMSPROP (torch.optim.RMSprop: sq = alpha sq + (1 - alpha) g^2, buf = momentum buf + g / (sqrt(sq) + eps), p -= lr buf; the
 * reference passes eps 1e-16, momentum 0.9, alpha is torch's default 0.99), GJ_OPT_ADAGRAD (sq += g^2, p -= lr g / (sqrt(sq) + eps),
 * eps 1e-16) and GJ_OPT_SGD (buf = momentum buf + g, p -= lr buf, momentum 0.9).  momentum_buf / sq_acc start at zero. */
#define GJ_OPT_RMSPROP 1
#define GJ_OPT_ADAGRAD 2
#define GJ_OPT_SGD 3
int gj_optimizer_step_flat(int32_t kind, float* param, const float* grad, float* momentum_buf, float* sq_acc, size_t n, float lr,
                           float alpha, float momentum, float eps, float grad_scale, float l1_lambda, float l2_lambda, void* stream);

/* sum|p| and sum p^2 over n floats into out[0], out[1] (overwritten; deterministic two-stage). */
int gj_param_norms(const float* param, size_t n, float* out, void* workspace, size_t workspace_bytes, void* stream);
size_t gj_param_norms_workspace(size_t n);

/* 'mean' latent map, encoder.py:147-149: y (B,N,W) -> z (B,W) and its adjoint. */
int gj_latent_mean_fwd(int32_t batch, int32_t num_nodes, int32_t width, const float* y, float* z, void* stream);
int gj_latent_mean_bwd(int32_t batch, int32_t num_nodes, int32_t width, const float* dz, float* dy, void* stream);

/* 'max' / 'min' latent maps (reference models/encoder.py:150-155: torch.amax / torch.amin over the particle axis):
 * z (batch,width) = extremum over n of y (batch,num_nodes,width); the adjoint shares dz evenly among the entries that attain the
 * extremum (torch's convention) and OVERWRITES dy. */
int gj_latent_extreme_fwd(int32_t batch, int32_t num_nodes, int32_t width, int32_t is_min, const float* y, float* z, void* stream);
int gj_latent_extreme_bwd(int32_t batch, int32_t num_nodes, int32_t width, const float* y, const float* z, const float* dz, float* dy,
                          void* stream);

/* Transform between the decoder's last step and the loss, y = clamp(tanh(x)) element by element over (rows, dim):
 * tanh if use_tanh (reference models/decoder.py:123-124, normalize_output), then a lower clamp at eps of the components whose bit
 * is set in clamp_mask (reference utils/train.py:55-65, polar coordinates: (E, pT) or pT).  The adjoint takes the untransformed x. */
int gj_output_transform_fwd(size_t rows, int32_t dim, int32_t use_tanh, int32_t clamp_mask, float eps, const float* x, float* y,
                            void* stream);
int gj_output_transform_bwd(size_t rows, int32_t dim, int32_t use_tanh, int32_t clamp_mask, float eps, const float* x, const float* dy,
                            float* dx, void* stream);

/* nn.MSELoss of reference utils/train.py:359-361 and its gradient: terms[0..1] = 0, terms[2] = sum (p - q)^2 / denom,
 * dp = 2 (p - q) / denom over `count` floats (denom = number of elements of the GLOBAL batch, so that data-parallel shards sum to the
 * single-device gradient).  Fixed summation order. */
size_t gj_mse_workspace(void);
int gj_mse_fwd_bwd(size_t count, double denom, const float* p, const float* q, float* terms, float* dp, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Small dense layer y = x W^T + b on the path's node/graph-level maps: decoder.py:127-136 (latent -> node
 * features) and the encoder mix layers, encoder.py:156-161.  x (rows,in), W (out,in) as nn.Linear, b (out) or
 * NULL, y (rows,out). */
int gj_linear_fwd(int32_t rows, int32_t in_f, int32_t out_f, const float* x, const float* w, const float* b,
                  float* y, void* stream);
size_t gj_linear_bwd_workspace(int32_t rows, int32_t in_f, int32_t out_f);
/* Adjoint: dx (rows,in) (may be NULL), dw (out,in) and db (out) (db may be NULL) OVERWRITTEN, fixed order. */
int gj_linear_bwd(int32_t rows, int32_t in_f, int32_t out_f, const float* x, const float* w, const float* dy,
                  float* dx, float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream);

/* Benchmark support (bench.py times the dominant kernel alone with these): relaunch ONLY the fused tensor-core edge
 * kernel of the step -- no node-level kernels, no reductions -- on the workspace that a preceding full gj_mp_step_fwd /
 * gj_mp_step_bwd call with the SAME arguments has populated (P|Q, pair distances, de, packed weights live there).
 * GJ_ERR_INVALID if the step does not run the fused tensor-core kernels (fp32 mode, other widths).  Results of the
 * backward relaunch are not meaningful (dQ accumulates onto the previous launch). */
int gj_bench_edge_fwd_only(const gj_mp_desc* d, const float* h, const float* params, float* e_out,
                           void* workspace, size_t workspace_bytes, void* stream);
int gj_bench_edge_bwd_only(const gj_mp_desc* d, const float* h, const float* params, float* dh, float* dparams,
                           void* workspace, size_t workspace_bytes, void* stream);
/* The same for the step as a training loop runs it: `saved` filled by gj_mp_step_fwd_saving, `workspace` by the
 * gj_mp_step_bwd_saved call that followed (the backward kernel then reads the saved P|Q, packed weights and pair distances). */
int gj_bench_edge_bwd_saved_only(const gj_mp_desc* d, const float* h, const float* params, float* dh, float* dparams,
                                 const void* saved, void* workspace, size_t workspace_bytes, void* stream);

/* Resource plan of the tensor-core (GJ_PREC_BF16) edge kernels for this step (host only, no device work):
 * info[0] forward shared-memory bytes per CTA, info[1] forward TMEM columns, info[2] backward shared-memory bytes
 * (0: these widths are not covered and the backward runs the fp32 kernel), info[3] backward TMEM columns. */
int gj_mp_plan_info(const gj_mp_desc* d, int32_t* info);

/* tcgen05 self-test: D(128 x n) = A(128 x k) * B(n x k)^T on one CTA with bf16 operands laid out
 * in the kernels' interleaved shared-memory layout; a_major/b_major: 0 = K-major, 1 = MN-major.
 * a_host_layout: A given as (128,k) row-major floats, B as (n,k) row-major floats (device pointers);
 * out receives the raw TMEM dump (128 lanes x n columns, row-major).  m is 64 or 128. */
int gj_umma_selftest(int32_t m, int32_t n, int32_t k, int32_t a_major, int32_t b_major,
                     const float* a, const float* b, float* out, void* stream);

/* The GEMM primitive of the generic-width node-level path (P|Q projections and node MLP of models/graphnet.py:249-271 at widths the
 * fused node kernels do not cover, e.g. BASELINE config 5's H = 64..256), exposed for testing.  Row-major fp32 tensors:
 *   form 0: C (M,N) = epi(A (M,K) . B (N,K)^T)      forward of a dense layer
 *   form 1: C (M,N) = epi(A (M,K) . B (K,N))        input gradient
 *   form 2: C (M,N) = A (K,M)^T . B (K,N)           weight gradient (split over K, fixed-order reduction; needs the workspace)
 * epi: + bias[n] (may be NULL), + previous C if accumulate, then act: 0 none, 1 LeakyReLU(alpha), 2 multiply by
 * (aux[m][n] > 0 ? 1 : alpha) (form 1 only); form 2 has no epilogue.  precision GJ_PREC_FP32: FFMA; GJ_PREC_BF16: tcgen05 (bf16 operands, fp32 accumulate). */
int gj_dense_gemm(int32_t form, int32_t M, int32_t N, int32_t K, const float* A, const float* B, const float* bias, int32_t act,
                  float alpha, const float* aux, int32_t accumulate, float* C, void* workspace, size_t workspace_bytes,
                  int32_t precision, void* stream);
size_t gj_dense_gemm_workspace(int32_t form, int32_t M, int32_t N, int32_t K);

/* Last error message of the calling thread ("" if none). */
const char* gj_last_error(void);

/* Library/ABI version and compiled architecture string, e.g. "sm_100a". */
int32_t gj_abi_version(void);
const char* gj_build_arch(void);

#ifdef __cplusplus
}
#endif
#endif /* GNNJET_B200_H */
