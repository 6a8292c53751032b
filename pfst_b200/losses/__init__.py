from .cross_entropy import decode_head_losses, upsample_cross_entropy
from .ohem import OHEMPixelSampler
from .pfgst_loss import PFGSTLoss, LOSS_KEYS

__all__ = ["PFGSTLoss", "LOSS_KEYS", "OHEMPixelSampler", "decode_head_losses", "upsample_cross_entropy"]
