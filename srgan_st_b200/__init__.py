"""srgan_st_b200 -- B200-native (sm_100a) loss hot path of SebastianBitsch/SRGAN-ST.

Public surface (mirrors reference loss.py): ``StructureTensorLoss``, ``BestBuddyLoss``, ``GramLoss``,
``PatchwiseStructureTensorLoss``; plus ``StructureTensorPixelLoss`` (ST + the "Pixel" MSE criterion fused) and
``structure_tensor_distance`` (the per-pixel ST distance map, differentiable).
Importing this package needs ``libsrst.so`` (build: ``python -m srgan_st_b200.build``); there is
no CPU or PyTorch fallback.
"""
from .loss import (BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss, StructureTensorLoss,  # noqa: F401
                   StructureTensorPixelLoss, structure_tensor_distance, structure_tensor_features)

__all__ = ["StructureTensorLoss", "BestBuddyLoss", "GramLoss", "PatchwiseStructureTensorLoss",
           "StructureTensorPixelLoss", "structure_tensor_distance", "structure_tensor_features"]
__version__ = "0.1.0"
