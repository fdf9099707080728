from .losses import BPRLoss, DualLoss, FullSoftmaxLoss, ListwiseLoss, SampledSoftmaxLoss, create_loss_function

__all__ = ["BPRLoss", "DualLoss", "FullSoftmaxLoss", "ListwiseLoss", "SampledSoftmaxLoss", "create_loss_function"]
