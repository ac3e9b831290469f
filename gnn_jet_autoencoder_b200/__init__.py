"""B200-native GraphNet message-passing path of the GNN jet autoencoder.

Drop-in surface (reference zichunhao/gnn-jet-autoencoder): ``GraphNet``, ``Encoder``, ``Decoder``
(models/), ``ChamferLoss`` (utils/losses/chamfer_loss), and ``GNNAETrainer`` -- the batch body of
utils/train.py:51-85 as one captured CUDA graph per step.  Everything executes in the sm_100a kernels
of ``libgnnjet_b200.so`` (C-ABI: include/gnnjet_b200.h); there is no CPU or eager fallback.
"""
from . import _lib
from .models import GraphNet, Encoder, Decoder
from .losses import ChamferLoss, EMDLoss, HungarianMSELoss
from .trainer import GNNAETrainer, synthetic_jets
from . import anomaly
from .permutation import PermutationTest

__all__ = ["GraphNet", "Encoder", "Decoder", "ChamferLoss", "EMDLoss", "HungarianMSELoss", "GNNAETrainer", "synthetic_jets", "anomaly",
           "PermutationTest", "_lib"]
