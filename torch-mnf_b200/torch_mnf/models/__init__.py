"""Models under the reference's public names (models/__init__.py:1-4).

MLP is the conditioner container of the coupling / spline flows (its Linear layers are packed into the flow program);
MNFLeNet and MNFFeedForward compose the MNF layers -- MNFLeNet.forward additionally drives the fused Monte-Carlo
pipeline (conv moments once per image, implicit-GEMM conv2, tensor-core fc1).  Both classifiers'
``predict_uncertainty`` return an MCUncertainty (predictive entropy, expected entropy, mutual information), finished
from device-side sums by ``uncertainty_from_sums``.  ``LeNet``, the deterministic comparison
network of the reference's README plot, is outside the hot path and not provided."""

from .mlp import MLP
from .mnf_feed_forward import MCUncertainty, MNFFeedForward, uncertainty_from_sums
from .mnf_lenet import MNFLeNet

__all__ = ["MLP", "MCUncertainty", "MNFFeedForward", "MNFLeNet", "uncertainty_from_sums"]
