"""B200-native supervised-contrastive (SupCon) loss path.

A from-scratch sm_100a implementation of the Stage-1 objective of
JaskiratSudan/wav2vec_contr_loss (``loss.py``), forward and backward, behind the
reference's own loss-class API.  PyTorch host code calls a thin C-ABI shared
library (``include/supcon_b200.h``) of hand-written CUDA kernels.
"""
from .loss import (BCEBinaryLoss, SupConBinaryLoss, SupConMultiClassLoss,  # noqa: F401
                   compute_pos_weight_from_dataset)
from .functional import l2_normalize, supcon_loss  # noqa: F401
from .head import FusedCompressionHead, layer_time_pool  # noqa: F401
from .memory import CrossBatchMemory, MemorySupConLoss  # noqa: F401

__version__ = "0.1.0"
