#!/usr/bin/env python
"""bf16-mode error of the whole model against the golden fixtures (GPU box): latent / reconstruction / concatenated gradient,
L2-relative, per golden case."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]
from test_gpu_parity import CASES, GOLDEN, DEV, build, gsub, make_input, rel  # noqa: E402
from gnn_jet_autoencoder_b200 import ChamferLoss  # noqa: E402

for name in sorted(CASES):
    case = CASES[name]
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    row = [name]
    for precision in ("fp32", "bf16"):
        enc, dec, ep, dp = build(case, precision)
        x = torch.from_numpy(make_input(case)).float().to(DEV)
        z = enc(x, metric=case["metric"])
        y = dec(z, metric=case["metric"])
        loss = ChamferLoss(case["loss_norm_choice"])(y, x, jet_features_weight=case["jet_features_weight"])
        (loss + case["l1_lambda"] * (enc.l1_norm() + dec.l1_norm())).backward()
        ne, nd = dict(enc.named_parameters()), dict(dec.named_parameters())
        eg = np.concatenate([ne[k].grad.cpu().numpy().ravel() for k in sorted(ep)])
        dg = np.concatenate([nd[k].grad.cpu().numpy().ravel() for k in sorted(dp)])
        row.append("%s: latent %.1e recon %.1e grad %.1e" % (
            precision, rel(z.detach().cpu().numpy(), g["latent"]), rel(y.detach().cpu().numpy(), g["recon"]),
            rel(np.concatenate([gsub(case, eg), gsub(case, dg)]), np.concatenate([g["enc_grad"], g["dec_grad"]]))))
    print("  ".join(row))
