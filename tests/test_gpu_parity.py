"""Parity of the CUDA path (through the C-ABI library) against the oracle and the reference-generated golden
vectors.  Tolerances (SURVEY.md 8.c / BASELINE north star):
  fp32 mode : <= 1e-5 L2-relative on latent, reconstruction, loss and the concatenated gradient
  bf16 mode : <= 2e-2 L2-relative on latent / reconstruction, <= 3e-2 on the concatenated gradient
"""
import os

import numpy as np
import pytest
import torch

import gnnae_oracle as O
from conftest import GOLDEN
from golden_cases import CASES, gsub, make_input, make_params
from gnn_jet_autoencoder_b200 import ChamferLoss, Decoder, Encoder, GNNAETrainer, GraphNet, _lib, ops
from gnn_jet_autoencoder_b200.trainer import synthetic_jets

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
TOL = {"fp32": dict(out=1e-5, grad=1e-5), "bf16": dict(out=2e-2, grad=3e-2)}


def rel(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def build(case, precision):
    ep, dp = make_params(case)
    enc = Encoder(**case["enc"], device=DEV, precision=precision)
    dec = Decoder(**case["dec"], device=DEV, precision=precision)
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in ep.items()})
    dec.load_state_dict({k: torch.from_numpy(v) for k, v in dp.items()})
    return enc, dec, ep, dp


# ---- tcgen05 building block ------------------------------------------------------------------------
def _tmem_rows(m):
    """TMEM lane of accumulator row r: M=128 -> lane r; M=64 -> rows sit in the first 16 lanes of each 32-lane
    quadrant."""
    if m == 128:
        return np.arange(128)
    return np.array([(r // 16) * 32 + (r % 16) for r in range(64)])


@pytest.mark.parametrize("m,n,k,a_mn,b_mn", [
    (128, 128, 32, 0, 0), (128, 64, 128, 0, 0), (128, 16, 64, 0, 0),      # forward layers (K-major x K-major)
    (128, 64, 16, 0, 1), (128, 128, 64, 0, 1), (128, 32, 128, 0, 1),      # dgrad (B = weights, MN-major view)
    (64, 16, 128, 1, 1), (128, 64, 128, 1, 1), (128, 32, 128, 1, 1),      # wgrad (both operands MN-major)
    (64, 32, 128, 0, 0),
])
def test_umma_selftest(m, n, k, a_mn, b_mn):
    g = torch.Generator().manual_seed(m + n + k)
    a = torch.randn(m, k, generator=g).to(torch.bfloat16).float()
    b = torch.randn(n, k, generator=g).to(torch.bfloat16).float()
    out = ops.umma_selftest(a.to(DEV), b.to(DEV), bool(a_mn), bool(b_mn)).cpu().numpy()
    want = (a.double() @ b.double().T).numpy()
    got = out[_tmem_rows(m)]
    assert rel(got, want) < 1e-5, (m, n, k, a_mn, b_mn, rel(got, want))


# ---- generic-width dense layer GEMM (node level at BASELINE config 5 widths) -------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("form,M,N,K", [
    (0, 300, 128, 256), (0, 129, 512, 3), (0, 1000, 20, 257), (0, 64, 256, 512),
    (1, 300, 256, 128), (1, 130, 3, 64), (1, 500, 513, 256),
    (0, 40000, 256, 256), (0, 38017, 72, 200), (1, 40000, 256, 256), (1, 38017, 130, 96),      # several hundred row tiles
    (2, 128, 256, 1000), (2, 256, 513, 700), (2, 20, 64, 129), (2, 3, 8, 5000),
])
def test_dense_gemm(form, M, N, K, precision):
    """C = A.B^T / A.B / A^T.B with the bias / LeakyReLU / slope-mask / accumulate epilogues against torch float64 (operands
    rounded to bf16 first in the bf16 mode, so the bound only has to cover the accumulation order)."""
    g = torch.Generator().manual_seed(form * 1000 + M + N + K)
    rnd = lambda *s: torch.randn(*s, generator=g)
    A = rnd(M, K) if form < 2 else rnd(K, M)
    B = rnd(N, K) if form == 0 else rnd(K, N)
    if precision == "bf16":
        A, B = A.to(torch.bfloat16).float(), B.to(torch.bfloat16).float()
    bias, aux, C0 = rnd(N), rnd(M, N), rnd(M, N)
    lib = _lib.load()
    prec = ops.PRECISIONS[precision]
    st = torch.cuda.current_stream().cuda_stream
    Ad, Bd = A.to(DEV), B.to(DEV)
    ws_bytes = lib.gj_dense_gemm_workspace(form, M, N, K)
    ws = torch.empty(ws_bytes // 4 + 16, device=DEV)
    ref = (A.double() @ B.double().T) if form == 0 else (A.double() @ B.double()) if form == 1 else (A.double().T @ B.double())
    # (bias, act, aux, accumulate): the bias / LeakyReLU epilogue belongs to the forward product, the slope mask to the input gradient
    cases = {0: [(None, 0, None, 0), (bias, 1, None, 0), (bias, 0, None, 1)], 1: [(None, 0, None, 0), (None, 2, aux, 0), (None, 0, None, 1)],
             2: [(None, 0, None, 0)]}[form]
    for b, act, ax, accum in cases:
        C = C0.clone().to(DEV)
        want = ref.clone()
        if b is not None:
            want = want + b.double()
        if accum:
            want = want + C0.double()
        if act == 1:
            want = torch.where(want > 0, want, 0.2 * want)
        elif act == 2:
            want = want * torch.where(ax > 0, 1.0, 0.2).double()
        bd = b.to(DEV) if b is not None else None
        axd = ax.to(DEV) if ax is not None else None
        _lib.check(lib.gj_dense_gemm(form, M, N, K, Ad.data_ptr(), Bd.data_ptr(), bd.data_ptr() if bd is not None else None, act, 0.2,
                                     axd.data_ptr() if axd is not None else None, accum, C.data_ptr(), ws.data_ptr(), ws_bytes, prec, st),
                   "gj_dense_gemm")
        torch.cuda.synchronize()
        assert rel(C.cpu().numpy(), want.numpy()) < 2e-6, (form, M, N, K, precision, act, accum, rel(C.cpu().numpy(), want.numpy()))


# ---- one message-passing step in isolation -----------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("N,H,edge,node,B,metric", [
    (30, 16, [32, 128, 64, 16], [16, 32], 3, "euclidean"),
    (6, 4, [32, 128, 64, 16], [4, 4], 5, "minkowskian"),      # fused tensor-core kernels with the Minkowskian distance
    (150, 32, [32, 128, 64, 16], [32, 8], 2, "euclidean"),     # five j blocks per jet (per-j-block partial sums)
    (31, 16, [32, 128, 64, 16], [16, 32], 3, "euclidean"),     # j-block boundaries of the fused kernels: 31 | 32 | 33 ...
    (32, 16, [32, 128, 64, 16], [16, 32], 3, "euclidean"),
    (64, 8, [32, 128, 64, 16], [8, 8], 2, "euclidean"),
    (96, 16, [32, 128, 64, 16], [16, 32], 1, "euclidean"),
    (160, 16, [32, 128, 64, 16], [16, 32], 1, "euclidean"),
    (30, 64, [64, 64], [64, 64], 3, "euclidean"),              # BASELINE config 5 shapes: edge [[H, H]], node [[H]]
    (33, 128, [128, 128], [128, 128], 2, "euclidean"),
    (9, 256, [256, 256], [256, 256], 2, "euclidean"),
    (5, 4, [16, 16], [4, 4], 7, "minkowskian"),
    (33, 8, [16, 32, 16], [8, 16, 8], 2, "euclidean"),
    (1, 3, [16], [3, 2], 4, "euclidean"),
    (64, 6, [8, 24], [6, 5], 2, "euclidean"),
    (10, 8, [16, 16], [180, 180], 3, "euclidean"),          # wide node MLP: V and V^T re-staged per GEMM, gradients in global partials
])
def test_mp_step_matches_oracle(precision, N, H, edge, node, B, metric):
    rng = np.random.default_rng(N * 100 + H)
    shapes_e = [(o, i) for i, o in zip([2 * H + 1] + edge[:-1], edge)]
    shapes_n = [(o, i) for i, o in zip([edge[-1] + H] + node[:-1], node)]
    ew = [rng.uniform(-1, 1, s) / np.sqrt(s[1]) for s in shapes_e]
    eb = [rng.uniform(-1, 1, s[0]) / np.sqrt(s[1]) for s in shapes_e]
    nw = [rng.uniform(-1, 1, s) / np.sqrt(s[1]) for s in shapes_n]
    nb = [rng.uniform(-1, 1, s[0]) / np.sqrt(s[1]) for s in shapes_n]
    h = rng.normal(0, 0.5, (B, N, H))
    dy = rng.normal(0, 1.0, (B, N, node[-1]))
    flat_ref = np.concatenate([np.concatenate([w.ravel(), b.ravel()]) for w, b in zip(ew, eb)] +
                              [np.concatenate([w.ravel(), b.ravel()]) for w, b in zip(nw, nb)])
    flat = torch.from_numpy(flat_ref).float().to(DEV)
    ht = torch.from_numpy(h).float().to(DEV)
    t = TOL[precision]
    # Random networks on random inputs put ~0.3 % of the pre-activations within bf16 rounding of the LeakyReLU kink; each
    # picks the other slope (an O(1) error on that element), which alone is sqrt(0.003) * 0.8 = 4 % of the step's gradient in
    # ANY bf16 evaluation order (measured 2e-2 .. 5.4e-2 on these cases).  The model-level golden tests (realistic weights /
    # jets) hold 3e-2.  The second pass, alpha = 1 (no kink, same kernels, same tiling / masking / reduction logic at the j-block
    # boundaries), isolates the arithmetic: gradients within 2e-2 (measured <= 7e-3).
    for alpha, gtol_bf16 in ((0.2, 8e-2), (1.0, 2e-2)):
        y_ref, cache = O.mp_step_forward(h, ew, eb, nw, nb, alpha, metric)
        dh_ref, dew, deb, dnw, dnb = O.mp_step_backward(dy, cache, ew, nw)
        gflat_ref = np.concatenate([np.concatenate([w.ravel(), b.ravel()]) for w, b in zip(dew, deb)] +
                                   [np.concatenate([w.ravel(), b.ravel()]) for w, b in zip(dnw, dnb)])
        args = (N, H, edge, node, alpha, ops.metric_id(metric), ops.PRECISIONS[precision])
        y, e = torch.ops.gnnjet.mp_step_fwd(ht, flat, *args)
        dh, dflat = torch.ops.gnnjet.mp_step_bwd(ht, e, flat, torch.from_numpy(dy).float().to(DEV), *args)
        gtol = t["grad"] if precision == "fp32" else gtol_bf16
        assert rel(y.cpu().numpy(), y_ref) < t["out"], alpha
        assert rel(e.cpu().numpy(), O.leaky(cache["edge_z"][-1], alpha).sum(axis=2)) < t["out"], alpha
        assert rel(dh.cpu().numpy(), dh_ref) < gtol, alpha
        assert rel(dflat.cpu().numpy(), gflat_ref) < gtol, alpha


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_wide_step_matches_oracle(precision):
    """H = 128 with a [128, 128] edge network (BASELINE config 5's middle width): the node level runs as generic GEMMs (dense.cu)
    in both modes; the edge network runs on the materialised, chunked edge path of dense.cu in fp32 (the fp32 edge kernels have
    no shared-memory plan for these widths) and on the third-generation fused kernels (edge3.cu) in bf16."""
    N, H, edge, node, B = 12, 128, [128, 128], [128, 8], 3
    rng = np.random.default_rng(128)
    shapes_e = [(o, i) for i, o in zip([2 * H + 1] + edge[:-1], edge)]
    shapes_n = [(o, i) for i, o in zip([edge[-1] + H] + node[:-1], node)]
    ew = [rng.uniform(-1, 1, s) / np.sqrt(s[1]) for s in shapes_e]
    eb = [rng.uniform(-1, 1, s[0]) / np.sqrt(s[1]) for s in shapes_e]
    nw = [rng.uniform(-1, 1, s) / np.sqrt(s[1]) for s in shapes_n]
    nb = [rng.uniform(-1, 1, s[0]) / np.sqrt(s[1]) for s in shapes_n]
    h = rng.normal(0, 0.5, (B, N, H))
    y_ref, cache = O.mp_step_forward(h, ew, eb, nw, nb, 0.2, "euclidean")
    pack = lambda ws, bs: [np.concatenate([w.ravel(), b.ravel()]) for w, b in zip(ws, bs)]
    flat = torch.from_numpy(np.concatenate(pack(ew, eb) + pack(nw, nb))).float().to(DEV)
    ht = torch.from_numpy(h).float().to(DEV)
    args = (N, H, edge, node, 0.2, 0, ops.PRECISIONS[precision])
    y, e = torch.ops.gnnjet.mp_step_fwd(ht, flat, *args)
    assert rel(y.cpu().numpy(), y_ref) < TOL[precision]["out"]
    assert rel(e.cpu().numpy(), O.leaky(cache["edge_z"][-1], 0.2).sum(axis=2)) < TOL[precision]["out"]
    dy = rng.normal(0, 1.0, y_ref.shape)
    dh_ref, dew, deb, dnw, dnb = O.mp_step_backward(dy, cache, ew, nw)
    gref = np.concatenate(pack(dew, deb) + pack(dnw, dnb))
    dh, dflat = torch.ops.gnnjet.mp_step_bwd(ht, e, flat, torch.from_numpy(dy).float().to(DEV), *args)
    gtol = 1e-5 if precision == "fp32" else 0.1      # bf16 forward, fp32 adjoint kernels: see test_mp_step_matches_oracle
    assert rel(dh.cpu().numpy(), dh_ref) < gtol
    assert rel(dflat.cpu().numpy(), gref) < gtol


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("alpha", [0.0, 1.0, 1.7])
def test_mp_step_alpha_range(precision, alpha):
    """LeakyReLU slopes at and beyond the edges of (0, 1): alpha > 1 takes the min(z, alpha z) form (the tensor-core
    kernels hand such steps to the fp32 kernels)."""
    rng = np.random.default_rng(7)
    N, H, edge, node, B = 12, 8, [32, 64, 16], [8, 6], 3
    shapes_e = [(o, i) for i, o in zip([2 * H + 1] + edge[:-1], edge)]
    shapes_n = [(o, i) for i, o in zip([edge[-1] + H] + node[:-1], node)]
    ew = [rng.uniform(-1, 1, s) / np.sqrt(s[1]) for s in shapes_e]
    eb = [rng.uniform(-1, 1, s[0]) / np.sqrt(s[1]) for s in shapes_e]
    nw = [rng.uniform(-1, 1, s) / np.sqrt(s[1]) for s in shapes_n]
    nb = [rng.uniform(-1, 1, s[0]) / np.sqrt(s[1]) for s in shapes_n]
    h = rng.normal(0, 0.5, (B, N, H))
    dy = rng.normal(0, 1.0, (B, N, node[-1]))
    y_ref, cache = O.mp_step_forward(h, ew, eb, nw, nb, alpha)
    dh_ref, dew, deb, dnw, dnb = O.mp_step_backward(dy, cache, ew, nw)
    pack = lambda ws, bs: [np.concatenate([w.ravel(), b.ravel()]) for w, b in zip(ws, bs)]
    flat = torch.from_numpy(np.concatenate(pack(ew, eb) + pack(nw, nb))).float().to(DEV)
    gref = np.concatenate(pack(dew, deb) + pack(dnw, dnb))
    ht = torch.from_numpy(h).float().to(DEV)
    args = (N, H, edge, node, alpha, 0, ops.PRECISIONS[precision])
    y, e = torch.ops.gnnjet.mp_step_fwd(ht, flat, *args)
    dh, dflat = torch.ops.gnnjet.mp_step_bwd(ht, e, flat, torch.from_numpy(dy).float().to(DEV), *args)
    tol = 1e-5 if precision == "fp32" else (2e-2 if alpha > 0 else 0.1)
    assert rel(y.cpu().numpy(), y_ref) < tol
    assert rel(dh.cpu().numpy(), dh_ref) < (1e-5 if precision == "fp32" else 0.1)
    assert rel(dflat.cpu().numpy(), gref) < (1e-5 if precision == "fp32" else 0.1)


# ---- whole model through the nn.Module (autograd) path, all golden cases --------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_modules_match_golden(name, precision):
    case = CASES[name]
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    enc, dec, ep, dp = build(case, precision)
    x = torch.from_numpy(make_input(case)).float().to(DEV)
    z = enc(x, metric=case["metric"])
    y = dec(z, metric=case["metric"])
    if case["polar_coord"]:      # the train loop's clamp (utils/train.py:55-65): plumbing around the modules
        k = 2 if y.shape[-1] == 4 else 1
        y = torch.cat([torch.clamp(y[..., :k], min=1e-16), y[..., k:]], dim=-1)
    crit = ChamferLoss(case["loss_norm_choice"])
    mse = case["loss_choice"] == "mse"
    loss = torch.nn.functional.mse_loss(y, x) if mse else crit(y, x, jet_features_weight=case["jet_features_weight"])
    total = loss + case["l1_lambda"] * (enc.l1_norm() + dec.l1_norm())
    total.backward()
    t = TOL[precision]
    assert tuple(z.shape) == g["latent"].shape and tuple(y.shape) == g["recon"].shape
    assert rel(z.detach().cpu().numpy(), g["latent"]) < t["out"]
    assert rel(y.detach().cpu().numpy(), g["recon"]) < t["out"]
    assert abs(total.item() - g["loss_intended"]) <= 2 * t["out"] * abs(g["loss_intended"]) + 1e-6
    if not mse:
        terms = crit.last_terms.cpu().numpy()
        assert abs(terms[0] - g["chamfer_term"]) <= 2 * t["out"] * abs(g["chamfer_term"]) + 1e-6
        assert abs(terms[1] - g["jet_term"]) <= 4 * t["out"] * abs(g["jet_term"]) + 1e-6
    ne, nd = dict(enc.named_parameters()), dict(dec.named_parameters())
    eg = np.concatenate([ne[k].grad.cpu().numpy().ravel() for k in sorted(ep)])
    dg = np.concatenate([nd[k].grad.cpu().numpy().ravel() for k in sorted(dp)])
    # arg-min ties can flip per-tensor gradients; the concatenated gradient is the stable quantity (SURVEY.md 7)
    assert rel(np.concatenate([gsub(case, eg), gsub(case, dg)]), np.concatenate([g["enc_grad"], g["dec_grad"]])) < t["grad"]
    # the value the reference actually returns (jet term only, chamfer_loss.py:42)
    ret = ChamferLoss(case["loss_norm_choice"], mode="reference")(y.detach(), x, jet_features_weight=case["jet_features_weight"])
    assert abs(ret.item() - g["returned"]) <= 4 * t["out"] * abs(g["returned"]) + 1e-6


# ---- fused trainer path ---------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["default_n30", "default_n33", "trainsh_n30", "local_mix_us_n8", "local_mix_sp_n8",
                                  "global_mix_n8", "bogus_map_n5", "mink_n6", "n1", "n2", "wide64_n9",
                                  "default_n31", "default_n32", "default_n64", "default_n150", "default_b257",
                                  "wide128_n30", "wide256_n12", "wide64_mps6_n10", "wide128_lat64_n33", "loss_mink3_n6",
                                  "max_n5", "min_n5", "broadcast_crop_n7", "mse_n6", "polar3_n6", "polar4_tanh_n6"])
@pytest.mark.parametrize("graph", [False, True])
def test_trainer_gradients_match_golden(name, precision, graph):
    case = CASES[name]
    if graph and name not in ("default_n30", "local_mix_us_n8"):
        pytest.skip("CUDA-graph replay is checked on two cases")
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    enc, dec, ep, dp = build(case, precision)
    tr = GNNAETrainer(enc, dec, batch_size=case["B"], loss_norm_choice=case["loss_norm_choice"],
                      jet_features_weight=case["jet_features_weight"], l1_lambda=case["l1_lambda"],
                      encoder_metric=case["metric"], decoder_metric=case["metric"], use_cuda_graph=graph,
                      loss_choice=case["loss_choice"], polar_coord=case["polar_coord"])
    x = torch.from_numpy(make_input(case)).float()
    tr.load_batch(x)
    tr.compute_gradients()
    tr.compute_gradients()      # second call replays the graph / re-runs: results must not accumulate
    torch.cuda.synchronize()
    t = TOL[precision]
    assert rel(tr.latent.cpu().numpy(), g["latent"]) < t["out"]
    assert rel(tr.recon.cpu().numpy(), g["recon"]) < t["out"]
    named = tr.named_gradients()
    sgn = lambda d: np.concatenate([np.sign(d[k]).ravel() for k in sorted(d)])
    # the L1 term is added inside the fused Adam
    got_e = np.concatenate([named["encoder." + k].cpu().numpy().ravel() for k in sorted(ep)]) + case["l1_lambda"] * sgn(ep)
    got_d = np.concatenate([named["decoder." + k].cpu().numpy().ravel() for k in sorted(dp)]) + case["l1_lambda"] * sgn(dp)
    assert rel(np.concatenate([gsub(case, got_e), gsub(case, got_d)]), np.concatenate([g["enc_grad"], g["dec_grad"]])) < t["grad"]
    stats = tr.stats.cpu().numpy()
    assert abs(tr.loss_from_stats(stats) - g["loss_intended"]) <= 2 * t["out"] * abs(g["loss_intended"]) + 1e-6


def test_trainer_step_matches_oracle_adam():
    """Three optimisation steps (fwd, Chamfer, bwd, fused flat Adam incl. L1 term) against the oracle's train_step."""
    case = CASES["trainsh_n30"]
    enc, dec, ep, dp = build(case, "fp32")
    lr = 1e-3
    tr = GNNAETrainer(enc, dec, batch_size=case["B"], lr=lr, use_cuda_graph=True)
    x = make_input(case)
    es, ds = {}, {}
    xt = torch.from_numpy(x).float().pin_memory()
    for _ in range(3):
        loss_ref, _, _ = O.train_step(x, ep, dp, case["enc"], case["dec"], es, ds, lr=lr)
        loss = tr.step(xt)
        assert abs(loss - loss_ref) <= 2e-5 * abs(loss_ref)
    for k, v in enc.state_dict().items():
        assert rel(v.cpu().numpy(), ep[k]) < 1e-5, k
    for k, v in dec.state_dict().items():
        assert rel(v.cpu().numpy(), dp[k]) < 1e-5, k


@pytest.mark.parametrize("graph", [False, True])
def test_run_epoch_equals_the_per_batch_loop(graph):
    """run_epoch (reference utils/train.py:51-120 without the per-batch host syncs) against step() batch by batch: same
    batch losses, same parameters, same collected outputs; the validation pass leaves the parameters untouched."""
    case = CASES["trainsh_n30"]
    B = case["B"]
    rng = np.random.default_rng(5)
    batches = [torch.from_numpy(make_input(case) * (1.0 + 0.1 * i) + rng.normal(0, 1e-3, make_input(case).shape)).float().pin_memory()
               for i in range(3)]
    enc_a, dec_a, _, _ = build(case, "fp32")
    enc_b, dec_b, _, _ = build(case, "fp32")
    tr_a = GNNAETrainer(enc_a, dec_a, batch_size=B, lr=1e-3, use_cuda_graph=graph)
    tr_b = GNNAETrainer(enc_b, dec_b, batch_size=B, lr=1e-3, use_cuda_graph=graph)
    losses, lat, rec = [], [], []
    for x in batches:
        losses.append(tr_a.step(x))
        lat.append(tr_a.latent.cpu().clone())
        rec.append(tr_a.recon.cpu().clone())
    avg, recons, targets, latents = tr_b.run_epoch(batches, is_train=True)
    assert abs(avg - sum(losses) / 3) <= 1e-6 * abs(avg)
    assert torch.equal(recons, torch.cat(rec)) and torch.equal(latents, torch.cat(lat))
    assert torch.equal(targets, torch.cat([b.reshape(tr_b.x.shape) for b in batches]))
    assert torch.equal(tr_a.flat, tr_b.flat)
    # validation: forward + loss only
    before = tr_b.flat.clone()
    vavg, vrec, _, _ = tr_b.run_epoch([b.to(DEV) for b in batches], is_train=False)
    assert torch.equal(tr_b.flat, before)
    tr_a.forward_only(batches[0])
    torch.cuda.synchronize()
    assert torch.equal(vrec[:B], tr_a.recon.cpu())
    assert np.isfinite(vavg) and vavg > 0
    # the training pass's collected outputs survive the validation pass (separate pinned caches per pass kind: the reference's
    # train_loop uses train()'s tensors after validate() has run, utils/train.py:196-236)
    assert torch.equal(recons, torch.cat(rec)) and torch.equal(latents, torch.cat(lat))
    with pytest.raises(ValueError):
        tr_b.run_epoch([batches[0][: B - 1]])


def test_float64_dtype_requests_keep_float32_parameters():
    """The reference's default flow builds the models with the CLI dtype float64 and runs PermutationTest(encoder, decoder,
    device, dtype=float64) before training (train.py:73-76, utils/permutation.py:19-20).  Parameters of the fused path stay
    float32 -- and keep their storage inside a live trainer's flat buffer -- while inputs / outputs follow the dtype."""
    from gnn_jet_autoencoder_b200 import PermutationTest
    case = CASES["trainsh_n30"]
    ep, dp = make_params(case)
    enc = Encoder(**case["enc"], device=DEV, dtype=torch.float64, precision="fp32")
    dec = Decoder(**case["dec"], device=DEV, dtype=torch.float64, precision="fp32")
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in ep.items()})
    dec.load_state_dict({k: torch.from_numpy(v) for k, v in dp.items()})
    tr = GNNAETrainer(enc, dec, batch_size=case["B"], use_cuda_graph=False)
    x64 = torch.from_numpy(make_input(case))
    out = PermutationTest(enc, dec, device=DEV, dtype=torch.float64)(x64)
    assert out["invariance"]["median"] < 1e-4      # 'mean' latent map: the autoencoder is permutation invariant
    assert all(p.dtype == torch.float32 for p in list(enc.parameters()) + list(dec.parameters()))
    assert enc.encoder._flat_ok() and dec.decoder._flat_ok()
    assert enc.encoder.edge_net[0][0].weight.data_ptr() == tr.flat.data_ptr()      # still a view of the trainer's buffer
    y = dec(enc(x64))
    assert y.dtype == torch.float64
    g = np.load(os.path.join(GOLDEN, "trainsh_n30.npz"))
    assert rel(y.detach().cpu().numpy(), g["recon"]) < 1e-5
    loss0 = tr.step(x64.float())
    assert np.isfinite(loss0)
    # moving the modules away breaks the views: forward must refuse instead of silently re-packing
    enc.cpu(); enc.to(DEV)
    with pytest.raises(RuntimeError):
        enc(x64)


# ---- permutation test harness (SURVEY 8.f rank 3) ----------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_permutation_test_on_the_cuda_modules(precision):
    """The GNNAE with the 'mean' latent map is permutation invariant (the decoder sees a permutation-invariant latent), so
    NN(P(x)) = NN(x) up to the summation order over j; the harness of utils/permutation.py reports it."""
    from gnn_jet_autoencoder_b200 import PermutationTest
    case = CASES["default_n30"]
    enc, dec, _, _ = build(case, precision)
    x = torch.from_numpy(make_input(case)).float()
    out = PermutationTest(enc, dec)(x)
    assert set(out) == {"invariance", "equivariance"}
    tol = 1e-4 if precision == "fp32" else 5e-2
    assert out["invariance"]["median"] < tol
    loader = torch.utils.data.DataLoader(x, batch_size=max(1, x.shape[0] // 2))
    out2 = PermutationTest(enc, dec, device=DEV, dtype=torch.float32)(loader, verbose=True)
    assert out2["invariance"]["values"].shape == (x.shape[0], case["enc"]["num_nodes"], 3)
    assert out2["invariance"]["median"] < tol


# ---- SURVEY 8.f components against the fixture the REFERENCE ITSELF produced (oracle/gen_golden_aux.py) ----------------
def test_anomaly_scores_match_the_reference_fixture():
    from gen_golden_aux import ANOMALY_SHAPES, aux_inputs
    from gnn_jet_autoencoder_b200 import anomaly
    g = np.load(os.path.join(GOLDEN, "aux_reference.npz"))
    for s, shape in enumerate(ANOMALY_SHAPES):
        p, q = aux_inputs(shape, s)
        pt, qt = torch.from_numpy(p).float().to(DEV), torch.from_numpy(q).float().to(DEV)
        tag = "x".join(map(str, shape))
        assert rel(anomaly.mse(pt, qt).cpu().numpy(), g[f"mse_{tag}"]) < 1e-6
        assert rel(anomaly.chamfer(pt, qt).cpu().numpy(), g[f"chamfer_{tag}"]) < 2e-5
        out_b = anomaly.chamfer(pt, qt, batch_size=2)
        assert not out_b.is_cuda and rel(out_b.numpy(), g[f"chamfer_b2_{tag}"]) < 2e-5      # the batched form returns a host tensor
        assert rel(anomaly.hungarian(pt, qt).cpu().numpy(), g[f"hungarian_{tag}"]) < 2e-5
        assert rel(anomaly.hungarian(pt, qt, batch_size=2).numpy(), g[f"hungarian_b2_{tag}"]) < 2e-5
        if shape[-1] == 4:
            assert rel(anomaly.chamfer_lorentz(pt, qt).cpu().numpy(), g[f"chamfer_lorentz_{tag}"]) < 5e-5
            assert rel(anomaly.hungarian_lorentz(pt, qt).cpu().numpy(), g[f"hungarian_lorentz_{tag}"]) < 2e-5


def test_hungarian_mse_loss_coordinate_modes_match_the_reference_fixture():
    """All four coordinate options of hungarian_mse.py:60-100; gradients where the reference can produce one (its relative modes
    raise under autograd)."""
    from gen_golden_aux import HUNGARIAN_MODES, aux_inputs
    from gnn_jet_autoencoder_b200 import HungarianMSELoss
    g = np.load(os.path.join(GOLDEN, "aux_reference.npz"))
    for s, shape in enumerate([(4, 30, 3), (3, 12, 4)]):
        p, q = aux_inputs(shape, 100 + s)
        for abs_coord, polar in HUNGARIAN_MODES:
            tag = "x".join(map(str, shape)) + f"_abs{int(abs_coord)}_polar{int(polar)}"
            pt = torch.from_numpy(p).to(DEV).requires_grad_(True)      # float64 in, as the reference's CLI default
            loss = HungarianMSELoss()(pt, torch.from_numpy(q).to(DEV), abs_coord=abs_coord, polar_coord=polar)
            assert abs(loss.item() - g[f"hmse_{tag}"]) <= 1e-6 * abs(g[f"hmse_{tag}"]), tag
            loss.backward()
            assert torch.isfinite(pt.grad).all()
            if abs_coord:
                assert rel(pt.grad.cpu().numpy(), g[f"hmse_grad_{tag}"]) < 1e-6, tag


# ---- anomaly-score distances (SURVEY 8.f rank 2) -----------------------------------------------------------
@pytest.mark.parametrize("B,N,D,lorentz", [(5, 30, 3, False), (3, 30, 4, False), (4, 30, 4, True), (2, 150, 4, True), (7, 1, 3, False),
                                            (300, 30, 3, False)])
def test_anomaly_chamfer_scores(B, N, D, lorentz):
    from gnn_jet_autoencoder_b200 import anomaly
    rng = np.random.default_rng(B * 7 + N)
    p, q = rng.normal(size=(B, N, D)).astype(np.float32), rng.normal(size=(B, N, D)).astype(np.float32)
    want = O.anomaly_chamfer(p.astype(np.float64), q.astype(np.float64), lorentz=lorentz)
    fn = anomaly.chamfer_lorentz if lorentz else anomaly.chamfer
    got = fn(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV))
    assert got.is_cuda and tuple(got.shape) == (B, N)
    assert np.allclose(got.cpu().numpy(), want, rtol=2e-5, atol=2e-5)
    got_b = fn(torch.from_numpy(p), torch.from_numpy(q), batch_size=2)          # batched form: host in, host out
    assert not got_b.is_cuda and torch.equal(got_b, got.cpu())
    assert torch.equal(anomaly.mse(torch.from_numpy(p), torch.from_numpy(q)), ((torch.from_numpy(p) - torch.from_numpy(q)) ** 2).sum(-1))
    with pytest.raises(RuntimeError):
        fn(torch.from_numpy(p).to(DEV), torch.from_numpy(q[:, : max(N - 1, 1)] if N > 1 else np.concatenate([q, q], 1)).to(DEV))


@pytest.mark.parametrize("B,N,D,lorentz", [(6, 30, 3, False), (4, 30, 4, True), (3, 150, 3, False), (2, 150, 4, True), (5, 1, 3, False),
                                            (5, 2, 4, False), (64, 33, 4, False)])
def test_anomaly_hungarian_matches_scipy(B, N, D, lorentz):
    """Device assignment solver against scipy.optimize.linear_sum_assignment (the reference's solver, through the oracle):
    same matching, same total cost, same (B, N) scores."""
    from gnn_jet_autoencoder_b200 import anomaly
    rng = np.random.default_rng(B * 13 + N)
    p, q = rng.normal(size=(B, N, D)).astype(np.float32), rng.normal(size=(B, N, D)).astype(np.float32)
    want, matching, total = O.anomaly_hungarian(p.astype(np.float64), q.astype(np.float64), lorentz=lorentz)
    m, t = anomaly.assignment(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV), lorentz=lorentz)
    m = m.cpu().numpy()
    assert all(sorted(row.tolist()) == list(range(N)) for row in m)
    assert np.allclose(t.cpu().numpy(), total, rtol=1e-5, atol=1e-4)          # optimal cost (the matching itself could differ on ties)
    assert np.array_equal(m, matching)
    fn = anomaly.hungarian_lorentz if lorentz else anomaly.hungarian
    got = fn(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV))
    assert tuple(got.shape) == (B, N) and np.allclose(got.cpu().numpy(), want, rtol=1e-5, atol=1e-5)
    got_b = fn(torch.from_numpy(p), torch.from_numpy(q), batch_size=3)
    assert not got_b.is_cuda and torch.allclose(got_b, got.cpu())


def test_hungarian_mse_loss_value_and_gradient():
    """HungarianMSELoss (hungarian_mse.py:27-58) against its lines written out with scipy + torch autograd on the host."""
    from scipy import optimize
    from gnn_jet_autoencoder_b200 import HungarianMSELoss
    rng = np.random.default_rng(21)
    p, q = rng.normal(size=(6, 30, 3)).astype(np.float32), rng.normal(size=(6, 30, 3)).astype(np.float32)
    ph = torch.from_numpy(p).requires_grad_(True)
    cost = torch.cdist(ph, torch.from_numpy(q)).detach().numpy()
    matching = [optimize.linear_sum_assignment(cost[i])[1] for i in range(len(cost))]
    shuffled = torch.stack([ph[i, torch.from_numpy(matching[i])] for i in range(len(matching))])
    want = torch.nn.MSELoss()(shuffled, torch.from_numpy(q))
    want.backward()
    pd = torch.from_numpy(p).to(DEV).requires_grad_(True)
    got = HungarianMSELoss()(pd, torch.from_numpy(q).to(DEV))
    got.backward()
    assert abs(got.item() - want.item()) <= 1e-6 * abs(want.item())
    assert torch.allclose(pd.grad.cpu(), ph.grad, rtol=1e-6, atol=1e-9)
    with pytest.raises(ValueError):
        HungarianMSELoss()(pd[..., :2], torch.from_numpy(q).to(DEV)[..., :2])


# ---- loss kernel ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,Np,Nq,D,norm", [(5, 30, 30, 3, "cartesian"), (3, 7, 11, 4, "minkowskian"), (2, 150, 150, 3, "cartesian"),
                                             (4, 1, 1, 4, "polar"), (300, 30, 30, 3, "polar")])
def test_chamfer_kernel(B, Np, Nq, D, norm):
    rng = np.random.default_rng(B + Np)
    p, q = rng.normal(size=(B, Np, D)), rng.normal(size=(B, Nq, D))
    p32, q32 = p.astype(np.float32).astype(np.float64), q.astype(np.float32).astype(np.float64)
    cham, jet, dcham, djet = O.chamfer_terms(p32, q32, norm)
    pt = torch.from_numpy(p).float().to(DEV).requires_grad_(True)
    crit = ChamferLoss(norm)
    loss = crit(pt, torch.from_numpy(q).float().to(DEV), jet_features_weight=0.5)
    loss.backward()
    terms = crit.last_terms.cpu().numpy()
    assert abs(terms[0] - cham) <= 1e-5 * abs(cham) + 1e-5 and abs(terms[1] - jet) <= 1e-5 * abs(jet) + 1e-5
    assert abs(loss.item() - (cham + 0.5 * jet)) <= 1e-5 * abs(cham + 0.5 * jet) + 1e-5
    assert rel(pt.grad.cpu().numpy(), dcham + 0.5 * djet) < 1e-5


def test_chamfer_errors_and_reference_mode():
    p = torch.zeros(2, 4, 3, device=DEV)
    with pytest.raises(ValueError):
        ChamferLoss("cartesian")(p, torch.zeros(3, 4, 3, device=DEV))
    with pytest.raises(ValueError):
        ChamferLoss("cartesian")(torch.zeros(2, 4, 5, device=DEV), torch.zeros(2, 4, 5, device=DEV))
    with pytest.raises(UnboundLocalError):
        ChamferLoss("cartesian", mode="reference")(p, p, jet_features_weight=0)
    # empty batch
    loss = ChamferLoss("cartesian")(torch.zeros(0, 4, 3, device=DEV), torch.zeros(0, 4, 3, device=DEV))
    assert loss.item() == 0.0


# ---- small kernels ---------------------------------------------------------------------------------------
def test_flat_adam_matches_torch():
    g = torch.Generator().manual_seed(0)
    p0 = torch.randn(10007, generator=g)
    p = p0.clone().to(DEV)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    ref = torch.nn.Parameter(p0.clone().double())
    opt = torch.optim.Adam([ref], 1e-3)
    for step in range(1, 6):
        gr = torch.randn(10007, generator=g)
        ops.adam_step_flat_(p, gr.to(DEV), m, v, step, lr=1e-3, l1_lambda=1e-3, l2_lambda=1e-2)
        ref.grad = gr.double() + 1e-3 * torch.sign(ref.detach()) + 2e-2 * ref.detach()
        opt.step()
    assert rel(p.cpu().numpy(), ref.detach().numpy()) < 1e-6


@pytest.mark.parametrize("kind", ["rmsprop", "adagrad", "sgd"])
def test_flat_optimizers_match_torch(kind):
    """gj_optimizer_step_flat against torch.optim with the hyper-parameters utils/initialize.py:154-170 passes."""
    g = torch.Generator().manual_seed(2)
    p0 = torch.randn(10007, generator=g)
    p = p0.clone().to(DEV)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    ref = torch.nn.Parameter(p0.clone().double())
    opt = {"rmsprop": lambda: torch.optim.RMSprop([ref], lr=1e-3, eps=1e-16, momentum=0.9),
           "adagrad": lambda: torch.optim.Adagrad([ref], lr=1e-3, eps=1e-16),
           "sgd": lambda: torch.optim.SGD([ref], lr=1e-3, momentum=0.9)}[kind]()
    for _ in range(5):
        gr = torch.randn(10007, generator=g)
        ops.optimizer_step_flat_(kind, p, gr.to(DEV), m, v, lr=1e-3, l1_lambda=1e-3, l2_lambda=1e-2)
        ref.grad = gr.double() + 1e-3 * torch.sign(ref.detach()) + 2e-2 * ref.detach()
        opt.step()
    assert rel(p.cpu().numpy(), ref.detach().numpy()) < 1e-6


def test_linear_and_latent_mean_and_norms():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(300, 20, generator=g).to(DEV).requires_grad_(True)
    w = torch.randn(48, 20, generator=g).to(DEV).requires_grad_(True)
    b = torch.randn(48, generator=g).to(DEV).requires_grad_(True)
    dy = torch.randn(300, 48, generator=g).to(DEV)
    ops.linear(x, w, b).backward(dy)
    x2, w2, b2 = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    torch.nn.functional.linear(x2, w2, b2).backward(dy.double())
    for a, r in ((x.grad, x2.grad), (w.grad, w2.grad), (b.grad, b2.grad)):
        assert rel(a.cpu().numpy(), r.cpu().numpy()) < 1e-5
    assert rel(ops.linear(x, w, None).detach().cpu().numpy(), (x2 @ w2.T).detach().cpu().numpy()) < 1e-5
    y = torch.randn(9, 30, 20, generator=g).to(DEV).requires_grad_(True)
    dz = torch.randn(9, 20, generator=g).to(DEV)
    z = ops.latent_mean(y)
    z.backward(dz)
    assert rel(z.detach().cpu().numpy(), y.detach().mean(1).cpu().numpy()) < 1e-6
    assert rel(y.grad.cpu().numpy(), (dz[:, None, :] / 30).expand(9, 30, 20).cpu().numpy()) < 1e-6
    n = ops.param_norms(w.detach().reshape(-1)).cpu().numpy()
    assert abs(n[0] - w.detach().abs().sum().item()) < 1e-3 and abs(n[1] - w.detach().pow(2).sum().item()) < 1e-3


# ---- properties at the BASELINE sizes (no oracle at this size) ----------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("N,B", [(30, 257), (150, 8)])
def test_permutation_equivariance_and_invariance(precision, N, B):
    """utils/permutation.py:76-109 semantics: GraphNet is equivariant, the 'mean' latent invariant."""
    from gnn_jet_autoencoder_b200.config import build_models
    enc, dec = build_models(N, device=DEV, precision=precision)
    x = torch.from_numpy(synthetic_jets(B, N, seed=3)).to(DEV)
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(0)).to(DEV)
    with torch.no_grad():
        y = enc.encoder(x)
        yp = enc.encoder(x[:, perm])
        z, zp = enc(x), enc(x[:, perm])
    tol = 1e-4 if precision == "fp32" else 5e-2
    assert rel(yp.cpu().numpy(), y[:, perm].cpu().numpy()) < tol
    assert rel(zp.cpu().numpy(), z.cpu().numpy()) < tol


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_full_size_step_is_deterministic_and_batch_linear(precision):
    """BASELINE config 2 size (N=30, B=4096): two runs give the same gradients -- bit-identical in fp32 mode; in bf16 mode
    the tile groups of a CTA add into shared TMEM weight-gradient accumulators in a timing-dependent order, so the runs
    agree to fp32 summation-order rounding -- and the gradient of the batch equals the sum of the gradients of its two
    halves (the loss is a sum over independent jets)."""
    from gnn_jet_autoencoder_b200.config import build_models
    N, B = 30, 4096
    x = torch.from_numpy(synthetic_jets(B, N, seed=11))
    grads = []
    for sl in (slice(0, B), slice(0, B), slice(0, B // 2), slice(B // 2, B)):
        enc, dec = build_models(N, device=DEV, precision=precision)
        tr = GNNAETrainer(enc, dec, batch_size=x[sl].shape[0], use_cuda_graph=False)
        tr.load_batch(x[sl])
        tr.compute_gradients()
        torch.cuda.synchronize()
        grads.append(tr.flat_gradient().clone())
        assert torch.isfinite(grads[-1]).all()
    if precision == "fp32":
        assert torch.equal(grads[0], grads[1])
    else:
        assert rel(grads[1].cpu().numpy(), grads[0].cpu().numpy()) < 1e-5
    assert rel((grads[2] + grads[3]).cpu().numpy(), grads[0].cpu().numpy()) < (1e-5 if precision == "fp32" else 1e-2)


def test_n150_forward_backward_runs_and_matches_fp32_vs_bf16():
    """BASELINE config 3 shape (N=150) at a small batch: bf16 tensor-core path against the fp32 path."""
    from gnn_jet_autoencoder_b200.config import build_models
    N, B = 150, 6
    x = torch.from_numpy(synthetic_jets(B, N, seed=5))
    out = {}
    for precision in ("fp32", "bf16"):
        enc, dec = build_models(N, device=DEV, precision=precision)
        tr = GNNAETrainer(enc, dec, batch_size=B, use_cuda_graph=False)
        tr.load_batch(x)
        tr.compute_gradients()
        torch.cuda.synchronize()
        out[precision] = (tr.recon.cpu().numpy().copy(), tr.flat_gradient().cpu().numpy().copy())
    assert rel(out["bf16"][0], out["fp32"][0]) < 2e-2
    assert rel(out["bf16"][1], out["fp32"][1]) < 3e-2


def test_saved_forward_byproducts_reproduce_the_plain_calls():
    """gj_mp_step_fwd_saving / gj_mp_step_bwd_saved (P|Q, packed weights and pair distances kept from forward) against
    gj_mp_step_fwd / gj_mp_step_bwd; steps that have nothing to save report 0 bytes and refuse the saving calls."""
    from gnn_jet_autoencoder_b200 import _lib
    lib = _lib.load()
    N, H, edge, node, B = 30, 16, [32, 128, 64, 16], [16, 32], 64
    rng = np.random.default_rng(3)
    npar = sum(o * i + o for i, o in zip([2 * H + 1] + edge[:-1], edge)) + sum(o * i + o for i, o in zip([edge[-1] + H] + node[:-1], node))
    flat = torch.from_numpy(rng.uniform(-0.3, 0.3, npar)).float().to(DEV)
    h = torch.from_numpy(rng.normal(0, 0.5, (B, N, H))).float().to(DEV)
    dy = torch.from_numpy(rng.normal(0, 1.0, (B, N, node[-1]))).float().to(DEV)
    d = _lib.make_desc(B, N, H, edge, node, 0.2, 0, ops.PRECISIONS["bf16"])
    nsaved = lib.gj_mp_step_saved_bytes(d)
    assert nsaved > 0
    ws_bytes = max(lib.gj_mp_step_fwd_workspace(d), lib.gj_mp_step_bwd_workspace(d))
    ws = torch.empty(ws_bytes // 4 + 1, device=DEV)
    saved = torch.empty(nsaved // 4 + 1, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    outs = []
    for use_saved in (False, True):
        y = torch.empty(B, N, node[-1], device=DEV); e = torch.empty(B, N, edge[-1], device=DEV)
        dh = torch.zeros(B, N, H, device=DEV); g = torch.empty(npar, device=DEV)
        sp = saved.data_ptr() if use_saved else None
        ops.raw_mp_fwd(d, h.data_ptr(), flat.data_ptr(), y.data_ptr(), e.data_ptr(), ws.data_ptr(), ws_bytes, st, sp)
        ops.raw_mp_bwd(d, h.data_ptr(), e.data_ptr(), flat.data_ptr(), dy.data_ptr(), dh.data_ptr(), g.data_ptr(), ws.data_ptr(), ws_bytes, st, sp)
        torch.cuda.synchronize()
        outs.append((y, e, dh, g))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert rel(outs[1][2].cpu().numpy(), outs[0][2].cpu().numpy()) < 1e-5
    assert rel(outs[1][3].cpu().numpy(), outs[0][3].cpu().numpy()) < 1e-5
    d32 = _lib.make_desc(B, N, H, edge, node, 0.2, 0, ops.PRECISIONS["fp32"])
    assert lib.gj_mp_step_saved_bytes(d32) == 0
    with pytest.raises(_lib.GnnJetError):
        ops.raw_mp_fwd(d32, h.data_ptr(), flat.data_ptr(), outs[0][0].data_ptr(), outs[0][1].data_ptr(), ws.data_ptr(), ws_bytes, st,
                       saved.data_ptr())


@pytest.mark.parametrize("shape", [([32, 128, 64, 16], [16, 32], 16), ([64, 64], [64], 64)])
def test_deterministic_mode_gives_bitwise_parameter_gradients(shape):
    """ops.set_deterministic (gj_set_deterministic): parameter gradients of the bf16 backward are bit-identical from run to run and
    agree with the default mode to fp32 summation order."""
    edge, node, H = shape
    N, B = 30, 1024
    rng = np.random.default_rng(11)
    npar = sum(o * i + o for i, o in zip([2 * H + 1] + edge[:-1], edge)) + sum(o * i + o for i, o in zip([edge[-1] + H] + node[:-1], node))
    flat = torch.from_numpy(rng.uniform(-0.2, 0.2, npar)).float().to(DEV)
    h = torch.from_numpy(rng.normal(0, 0.5, (B, N, H))).float().to(DEV)
    dy = torch.from_numpy(rng.normal(0, 1.0, (B, N, node[-1]))).float().to(DEV)
    args = (N, H, edge, node, 0.2, 0, ops.PRECISIONS["bf16"])
    y, e = torch.ops.gnnjet.mp_step_fwd(h, flat, *args)
    dh0, g0 = torch.ops.gnnjet.mp_step_bwd(h, e, flat, dy, *args)
    prev = ops.set_deterministic(True)
    try:
        runs = [torch.ops.gnnjet.mp_step_bwd(h, e, flat, dy, *args) for _ in range(3)]
    finally:
        ops.set_deterministic(prev)
    torch.cuda.synchronize()
    for dh, g in runs[1:]:
        assert torch.equal(g, runs[0][1]) and torch.equal(dh, runs[0][0])
    # against the default mode: same sums in a different grouping (the tile ranges of the groups differ)
    assert rel(runs[0][0].cpu().numpy(), dh0.cpu().numpy()) < 1e-5
    assert rel(runs[0][1].cpu().numpy(), g0.cpu().numpy()) < 1e-5


@pytest.mark.parametrize("N,B", [(30, 64), (33, 9)])
def test_batched_pack_and_deferred_reduction_match_the_per_step_calls(N, B):
    """gj_mp_steps_pack / gj_mp_step_fwd_packed / gj_mp_step_bwd_deferred / gj_mp_steps_reduce (one packing launch and one
    reduction launch per training step) against the per-step gj_mp_step_fwd_saving / gj_mp_step_bwd_saved path: same summation
    order, so -- in the deterministic mode, which fixes the order inside the backward edge kernel -- the flat gradient is
    bit-identical; forward outputs and the loss are bit-identical in any mode."""
    from gnn_jet_autoencoder_b200 import GNNAETrainer, synthetic_jets
    from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models
    x = torch.from_numpy(synthetic_jets(B, N, seed=21))
    prev = ops.set_deterministic(True)
    try:
        res = []
        for batched in (False, True):
            enc, dec = build_models(N, DEFAULT_ARCH, device=DEV, precision="bf16", seed=4)
            tr = GNNAETrainer(enc, dec, batch_size=B, use_cuda_graph=False, batched_launches=batched)
            assert tr.batched == batched
            before = ops.LAUNCHES["count"]
            tr.load_batch(x)
            tr.compute_gradients()
            torch.cuda.synchronize()
            res.append((tr.grad.clone(), tr.latent.clone(), tr.recon.clone(), tr.stats.clone(), ops.LAUNCHES["count"] - before))
    finally:
        ops.set_deterministic(prev)
    (g0, z0, r0, s0, n0), (g1, z1, r1, s1, n1) = res
    assert torch.equal(z0, z1) and torch.equal(r0, r1) and torch.equal(s0, s1)
    assert torch.equal(g0, g1)
    assert float(g0.abs().sum()) > 0
    assert n1 == n0 - 10      # six packing launches -> one, six reductions -> one


def test_bench_hooks_relaunch_the_fused_kernels():
    """gj_bench_edge_*_only (bench.py's roofline timing) run on the workspace of a preceding full call; the forward
    relaunch reproduces e bit for bit; steps outside the fused kernels are refused."""
    lib = _lib.load()
    N, H, edge, node, B = 30, 16, [32, 128, 64, 16], [16, 32], 16
    npar = sum(o * i + o for i, o in zip([2 * H + 1] + edge[:-1], edge)) + sum(o * i + o for i, o in zip([edge[-1] + H] + node[:-1], node))
    g = torch.Generator(device="cpu").manual_seed(5)
    flat = ((torch.rand(npar, generator=g) - 0.5) * 0.4).to(DEV)
    h = (torch.randn(B, N, H, generator=g) * 0.5).to(DEV)
    dy = torch.randn(B, N, node[-1], generator=g).to(DEV)
    d = _lib.make_desc(B, N, H, edge, node, 0.2, 0, ops.PRECISIONS["bf16"])
    ws_bytes = max(lib.gj_mp_step_fwd_workspace(d), lib.gj_mp_step_bwd_workspace(d))
    ws = torch.empty(ws_bytes // 4 + 1, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    y = torch.empty(B, N, node[-1], device=DEV); e = torch.empty(B, N, edge[-1], device=DEV); e2 = torch.zeros_like(e)
    dh = torch.zeros(B, N, H, device=DEV); gr = torch.empty(npar, device=DEV)
    ops.raw_mp_fwd(d, h.data_ptr(), flat.data_ptr(), y.data_ptr(), e.data_ptr(), ws.data_ptr(), ws_bytes, st)
    assert lib.gj_bench_edge_fwd_only(d, h.data_ptr(), flat.data_ptr(), e2.data_ptr(), ws.data_ptr(), ws_bytes, st) == 0
    torch.cuda.synchronize()
    assert torch.equal(e, e2)
    ops.raw_mp_bwd(d, h.data_ptr(), e.data_ptr(), flat.data_ptr(), dy.data_ptr(), dh.data_ptr(), gr.data_ptr(), ws.data_ptr(), ws_bytes, st)
    assert lib.gj_bench_edge_bwd_only(d, h.data_ptr(), flat.data_ptr(), dh.data_ptr(), gr.data_ptr(), ws.data_ptr(), ws_bytes, st) == 0
    torch.cuda.synchronize()
    d32 = _lib.make_desc(B, N, H, edge, node, 0.2, 0, ops.PRECISIONS["fp32"])
    assert lib.gj_bench_edge_fwd_only(d32, h.data_ptr(), flat.data_ptr(), e2.data_ptr(), ws.data_ptr(), ws_bytes, st) != 0


def test_module_path_equals_trainer_path():
    case = CASES["default_n30"]
    enc, dec, ep, dp = build(case, "fp32")
    x = torch.from_numpy(make_input(case)).float().to(DEV)
    loss = ChamferLoss("cartesian")(dec(enc(x)), x)
    loss.backward()
    ge = {k: p.grad.clone() for k, p in enc.named_parameters()}
    tr = GNNAETrainer(enc, dec, batch_size=case["B"], use_cuda_graph=False)
    tr.load_batch(x)
    tr.compute_gradients()
    torch.cuda.synchronize()
    named = tr.named_gradients()
    for k, v in ge.items():
        assert torch.allclose(named["encoder." + k], v, rtol=1e-5, atol=1e-7), k


def test_bad_arguments_raise():
    flat = torch.zeros(10, device=DEV)
    with pytest.raises(_lib.GnnJetError):
        torch.ops.gnnjet.mp_step_fwd(torch.zeros(1, 4, 3, device=DEV), flat, 4, 3, [8], [3], 0.2, 0, 0)
    g = GraphNet(4, 3, 2, [[4]], [[8]], 1, dropout=0.5, device=DEV)
    with pytest.raises(NotImplementedError):
        g(torch.zeros(1, 4, 3, device=DEV))
