"""The oracle against the reference's own outputs (tests/golden/, produced by
oracle/gen_golden.py running the unmodified reference in float64)."""
import json
import os

import numpy as np
import pytest

import gnnae_oracle as O
from golden_cases import CASES, gsub, make_input, make_params
from conftest import GOLDEN


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64).ravel() - np.asarray(b, np.float64).ravel())
                 / (np.linalg.norm(np.asarray(b, np.float64).ravel()) + 1e-300))


def test_index_lists_every_case():
    idx = json.load(open(os.path.join(GOLDEN, "index.json")))
    assert sorted(idx["cases"]) == sorted(CASES)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference(name):
    case = CASES[name]
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    ep, dp = make_params(case)
    x = make_input(case)
    loss, z, y, eg, dg = O.loss_and_grads(
        x, ep, dp, case["enc"], case["dec"], metric=case["metric"], loss_norm_choice=case["loss_norm_choice"],
        jet_features_weight=case["jet_features_weight"], l1_lambda=case["l1_lambda"], loss_choice=case["loss_choice"],
        polar_coord=case["polar_coord"])
    tol = 1e-12 if case["store64"] else 2e-7   # float32-stored fixtures carry 6e-8 rounding
    assert z.shape == g["latent"].shape and y.shape == g["recon"].shape
    assert rel(z, g["latent"]) < 1e-12
    assert rel(y, g["recon"]) < 1e-12
    assert abs(loss - g["loss_intended"]) <= 1e-11 * abs(g["loss_intended"])
    egf = np.concatenate([eg[k].ravel() for k in sorted(ep)])
    dgf = np.concatenate([dg[k].ravel() for k in sorted(dp)])
    assert rel(gsub(case, egf), g["enc_grad"]) < tol
    assert rel(gsub(case, dgf), g["dec_grad"]) < tol
    # the value the reference actually returns (jet term only) and the two terms separately
    cham, jet, _, _ = O.chamfer_terms(y, x, case["loss_norm_choice"])
    assert abs(cham - g["chamfer_term"]) <= 1e-11 * max(1.0, abs(g["chamfer_term"]))
    assert abs(jet - g["jet_term"]) <= 1e-11 * max(1.0, abs(g["jet_term"]))
    ret, _ = O.chamfer_loss(y, x, case["loss_norm_choice"], case["jet_features_weight"], mode="reference")
    assert abs(ret - g["returned"]) <= 1e-11 * max(1.0, abs(g["returned"]))


def test_reference_mode_raises_on_zero_weight():
    x = O.synthetic_jets(2, 5, dtype=np.float64)
    with pytest.raises(UnboundLocalError):
        O.chamfer_loss(x, x[:, ::-1], jet_features_weight=0, mode="reference")


def test_pairwise_distance_validation():
    p = np.zeros((2, 4, 3))
    with pytest.raises(ValueError):
        O.pairwise_distance_sq(p, np.zeros((3, 4, 3)))
    with pytest.raises(ValueError):
        O.pairwise_distance_sq(np.zeros((2, 4, 5)), np.zeros((2, 4, 5)))
    with pytest.raises(ValueError):
        O.pairwise_distance_sq(p, np.zeros((2, 4, 4)))


def test_adjust_var_list_semantics():
    assert O.adjust_var_list([[1], [2]], 4) == [[1], [2], [2], [2]]
    assert O.adjust_var_list([[1], [2], [3]], 2) == [[1], [2]]
    assert O.adjust_var_list(0.2, 3) == [0.2, 0.2, 0.2]


def test_backward_matches_finite_differences():
    rng = np.random.default_rng(0)
    case = CASES["max_n5"]
    ep, dp = make_params(case)
    x = make_input(case)
    kw = dict(metric="euclidean", l1_lambda=0.0)
    loss, *_, eg, dg = O.loss_and_grads(x, ep, dp, case["enc"], case["dec"], **kw)
    for params, grads in ((ep, eg), (dp, dg)):
        for k in list(params)[::3]:
            idx = tuple(rng.integers(0, s) for s in params[k].shape)
            old = params[k][idx]
            h = 1e-6
            params[k][idx] = old + h
            lp = O.loss_and_grads(x, ep, dp, case["enc"], case["dec"], **kw)[0]
            params[k][idx] = old - h
            lm = O.loss_and_grads(x, ep, dp, case["enc"], case["dec"], **kw)[0]
            params[k][idx] = old
            fd = (lp - lm) / (2 * h)
            assert abs(fd - grads[k][idx]) <= 1e-5 * max(1.0, abs(fd)), (k, idx, fd, grads[k][idx])


def test_permutation_equivariance_of_oracle():
    """utils/permutation.py:76-109 semantics: decoder(encoder(Px)) vs P decoder(encoder(x)) for the
    per-node ('local mix') map, and invariance of the latent for 'mean'."""
    case = CASES["local_mix_us_n8"]
    ep, dp = make_params(case)
    x = make_input(case)
    perm = np.random.default_rng(1).permutation(case["N"])
    z, _ = O.encoder_forward(x, ep, case["enc"])
    y, _ = O.decoder_forward(z, dp, case["dec"])
    zp, _ = O.encoder_forward(x[:, perm], ep, case["enc"])
    yp, _ = O.decoder_forward(zp, dp, case["dec"])
    assert O.relative_deviation(yp, y[:, perm]).max() < 1e-9
    case = CASES["trainsh_n30"]
    ep, dp = make_params(case)
    x = make_input(case)
    perm = np.random.default_rng(2).permutation(case["N"])
    z, _ = O.encoder_forward(x, ep, case["enc"])
    zp, _ = O.encoder_forward(x[:, perm], ep, case["enc"])
    assert np.abs(zp - z).max() < 1e-12


def test_adam_matches_torch():
    import torch
    rng = np.random.default_rng(3)
    p0 = rng.normal(size=(7, 5))
    params = {"w": p0.copy()}
    state = {}
    tp = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    opt = torch.optim.Adam([tp], 1e-3)
    for _ in range(5):
        g = rng.normal(size=p0.shape)
        O.adam_update(params, {"w": g}, state, lr=1e-3)
        tp.grad = torch.from_numpy(g.copy())
        opt.step()
    assert np.abs(params["w"] - tp.detach().numpy()).max() < 1e-14


@pytest.mark.parametrize("name", ["default_n30", "trainsh_n30", "local_mix_sp_n8", "global_mix_n8", "max_n5", "mink_n6",
                                  "broadcast_crop_n7", "n1"])
def test_torch_port_matches_reference(name):
    """oracle/torch_port.py (the CPU-baseline restatement timed by bench.py) against the reference's outputs."""
    import torch
    import torch_port as TP
    case = CASES[name]
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    ep, dp = make_params(case)
    x = torch.from_numpy(make_input(case))
    tep, tdp = TP.make_params(ep, torch.float64), TP.make_params(dp, torch.float64)
    loss, z, y = TP.loss_fn(x, tep, tdp, case["enc"], case["dec"], metric=case["metric"],
                            loss_norm_choice=case["loss_norm_choice"], jet_features_weight=case["jet_features_weight"],
                            l1_lambda=case["l1_lambda"])
    loss.backward()
    assert rel(z.detach().numpy(), g["latent"]) < 1e-12
    assert rel(y.detach().numpy(), g["recon"]) < 1e-12
    assert abs(loss.item() - g["loss_intended"]) <= 1e-11 * abs(g["loss_intended"])
    eg = np.concatenate([tep[k].grad.numpy().ravel() for k in sorted(ep)])
    dg = np.concatenate([tdp[k].grad.numpy().ravel() for k in sorted(dp)])
    tol = 1e-11 if case["store64"] else 2e-7
    assert rel(gsub(case, eg), g["enc_grad"]) < tol and rel(gsub(case, dg), g["dec_grad"]) < tol


def test_anomaly_chamfer_against_a_torch_restatement():
    """anomaly_detection.py:482-488 / :505-510 written out with torch (the module itself needs energyflow / jetnet /
    matplotlib and is not importable here): the oracle's numpy form gives the same (B, N) scores."""
    import torch
    rng = np.random.default_rng(3)
    p, q = rng.normal(size=(4, 9, 4)), rng.normal(size=(4, 9, 4))
    pt, qt = torch.from_numpy(p), torch.from_numpy(q)
    diffs = torch.unsqueeze(pt, -2) - torch.unsqueeze(qt, -3)
    dist = torch.norm(diffs, dim=-1)
    want = torch.min(dist, dim=-1).values + torch.min(dist, dim=-2).values
    assert np.allclose(O.anomaly_chamfer(p, q), want.numpy(), rtol=1e-12, atol=0)
    E, px, py, pz = diffs.unbind(-1)
    dl = E ** 2 - px ** 2 - py ** 2 - pz ** 2
    want_l = torch.min(dl, dim=-1).values + torch.min(dl, dim=-2).values
    assert np.allclose(O.anomaly_chamfer(p, q, lorentz=True), want_l.numpy(), rtol=1e-12, atol=0)
    assert O.anomaly_chamfer(p[..., :3], q[..., :3]).shape == (4, 9)


def test_anomaly_hungarian_oracle_properties():
    """The oracle's matching is scipy's (the reference's solver): a permutation per jet, never worse than the identity or a
    random matching, and exact on a permuted copy (score 0, matching = inverse permutation)."""
    rng = np.random.default_rng(11)
    p = rng.normal(size=(5, 8, 4))
    perm = np.stack([rng.permutation(8) for _ in range(5)])
    q = p[np.arange(5)[:, None], perm]                       # q_j = p_perm[j]
    score, matching, total = O.anomaly_hungarian(p, q)
    assert np.allclose(total, 0) and np.allclose(p[np.arange(5)[:, None], matching], p[np.arange(5)[:, None], matching])
    assert all(sorted(m.tolist()) == list(range(8)) for m in matching)
    inv = np.argsort(perm, axis=1)                            # row i of p sits at column inv[i] of q
    assert np.array_equal(matching, inv)
    q2 = rng.normal(size=(5, 8, 4))
    _, m2, t2 = O.anomaly_hungarian(p, q2, lorentz=True)
    d = p[:, :, None, :] - q2[:, None, :, :]
    c = d[..., 0] ** 2 - (d[..., 1:] ** 2).sum(-1)
    assert np.all(t2 <= np.trace(c, axis1=1, axis2=2) + 1e-12)



# ---- SURVEY 8.f components against fixtures produced by the reference itself (oracle/gen_golden_aux.py) ----------------
def _aux():
    return np.load(os.path.join(GOLDEN, "aux_reference.npz"))


def test_anomaly_scores_match_the_reference_fixture():
    """mse / chamfer / chamfer_lorentz / hungarian / hungarian_lorentz of utils/jet_analysis/anomaly_detection.py:454-590, plain
    and batched: the numpy oracle equals the outputs of the imported reference module."""
    from gen_golden_aux import ANOMALY_SHAPES, aux_inputs
    g = _aux()
    for s, shape in enumerate(ANOMALY_SHAPES):
        p, q = aux_inputs(shape, s)
        tag = "x".join(map(str, shape))
        assert np.allclose(((p - q) ** 2).sum(-1), g[f"mse_{tag}"], rtol=1e-13)
        for key in (f"chamfer_{tag}", f"chamfer_b2_{tag}"):
            assert rel(O.anomaly_chamfer(p, q), g[key]) < 1e-13
        for key in (f"hungarian_{tag}", f"hungarian_b2_{tag}"):
            assert rel(O.anomaly_hungarian(p, q)[0], g[key]) < 1e-13
        if shape[-1] == 4:
            assert rel(O.anomaly_chamfer(p, q, lorentz=True), g[f"chamfer_lorentz_{tag}"]) < 1e-13
            assert rel(O.anomaly_hungarian(p, q, lorentz=True)[0], g[f"hungarian_lorentz_{tag}"]) < 1e-13


def test_hungarian_mse_coordinate_modes_match_the_reference_fixture():
    from gen_golden_aux import HUNGARIAN_MODES, aux_inputs
    g = _aux()
    for s, shape in enumerate([(4, 30, 3), (3, 12, 4)]):
        p, q = aux_inputs(shape, 100 + s)
        for abs_coord, polar in HUNGARIAN_MODES:
            tag = "x".join(map(str, shape)) + f"_abs{int(abs_coord)}_polar{int(polar)}"
            assert abs(O.hungarian_mse_loss(p, q, abs_coord, polar) - g[f"hmse_{tag}"]) <= 1e-12 * abs(g[f"hmse_{tag}"]), tag


def test_hungarian_coordinate_maps_of_the_package_match_the_oracle():
    """The product's torch coordinate maps (CPU tensors are fine here: only the matching needs the GPU) against the oracle."""
    import torch
    from gen_golden_aux import HUNGARIAN_MODES, aux_inputs
    from gnn_jet_autoencoder_b200.losses import hungarian_preprocess
    for s, shape in enumerate([(4, 30, 3), (3, 12, 4)]):
        p, q = aux_inputs(shape, 100 + s)
        for abs_coord, polar in HUNGARIAN_MODES:
            r, t = hungarian_preprocess(torch.from_numpy(p), torch.from_numpy(q), abs_coord, polar)
            ro, to = O.hungarian_coords(p, q, abs_coord, polar)
            assert rel(r.numpy(), ro) < 1e-13 and rel(t.numpy(), to) < 1e-13


def test_permutation_helpers_match_the_reference_fixture():
    import torch
    from gnn_jet_autoencoder_b200.permutation import apply_perm, dev
    g = _aux()
    x, perm = torch.from_numpy(g["perm_x"]), torch.from_numpy(g["perm_perm"])
    assert np.array_equal(apply_perm(perm, x).numpy(), g["perm_apply"])
    assert np.allclose(dev(x, torch.from_numpy(g["perm_x"][:, ::-1].copy())).numpy(), g["perm_dev"], rtol=1e-13)


def test_modules_take_the_reference_checkpoint_layout(tmp_path):
    """The package's Encoder / Decoder with the reference's CLI-default architecture (N=30, dtype float64 requested as the CLI
    does) carry the reference's state_dict: the names and shapes of the default_n30 fixture parameters, which oracle/gen_golden.py
    loaded strictly into the reference's own modules, and the parameter counts of the reference's gradients in
    tests/golden/index.json.  A float64 checkpoint in that layout, saved and read back the way utils/initialize.py:54-128 does for
    --load-to-train, loads into the new modules as float32; their state_dicts load into modules of the same layout; an optimiser
    over their parameters covers every learnable parameter."""
    import torch
    from gnn_jet_autoencoder_b200 import Decoder, Encoder
    case = CASES["default_n30"]
    counts = json.load(open(os.path.join(GOLDEN, "index.json")))["cases"]["default_n30"]
    ep, dp = make_params(case)
    mk = lambda: (Encoder(**case["enc"], device="cpu", dtype=torch.float64), Decoder(**case["dec"], device="cpu", dtype=torch.float64))
    enc, dec = mk()
    for new, ref, n in ((enc, ep, counts["n_enc"]), (dec, dp, counts["n_dec"])):
        assert {k: tuple(v.shape) for k, v in new.state_dict().items()} == {k: v.shape for k, v in ref.items()}
        assert new.num_learnable_params == n
        opt = torch.optim.Adam(new.parameters(), lr=1e-3)
        assert sum(p.numel() for g in opt.param_groups for p in g["params"]) == n
    for side, new, ref in (("encoder", enc, ep), ("decoder", dec, dp)):
        path = tmp_path / f"weights_{side}" / f"epoch_3_{side}_weights.pth"
        path.parent.mkdir()
        torch.save({k: torch.from_numpy(v.astype(np.float64)) for k, v in ref.items()}, path)
        new.load_state_dict(torch.load(path, map_location=torch.device("cpu")))
        for k, v in new.state_dict().items():
            assert v.dtype == torch.float32 and np.array_equal(v.numpy(), ref[k].astype(np.float64).astype(np.float32))
    enc2, dec2 = mk()
    enc2.load_state_dict(enc.state_dict()); dec2.load_state_dict(dec.state_dict())
    for a, b in ((enc2, enc), (dec2, dec)):
        assert all(torch.equal(v, b.state_dict()[k]) for k, v in a.state_dict().items())
