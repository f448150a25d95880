"""ctunet_b200 -- B200-native (sm_100a) implementation of the 3D U-Net hot path of vfmatzkin/ct-unet.

Public surface mirrors the reference's (``ctunet.pytorch.models``, ``ctunet.utilities.dice_loss`` /
``hard_segm_from_tensor``, the ``comp_losses_metrics`` handlers); see INTEGRATION.md for how it plugs
into the reference's ``Model`` class.
"""
from . import _lib  # noqa: F401
from .models import (UNet, UNet4b1i3o, UNet4b2i3o, UNet5b2i3o, UNetDO, UNetSP, UNetSPSmall, UNet4_2IC,  # noqa: F401
                     recAE_v2_fixed, UNetBlock, CenterBlock, ResidualBlock, down_block_cr, up_block_cr,
                     set_compute_dtype, get_compute_dtype)
from .losses import (dice_loss, dice_ce, ProblemHandler, FlapRec, FlapRecWithShapePrior,  # noqa: F401
                     FlapRecWithShapePriorDoubleOut, FlapRecDoubleOut)
from .utilities import (hard_segm_from_tensor, shape_3d, blank_patch, random_blank_patch, encode_flaprec_batch,  # noqa: F401
                        SkullRandomHole, SaltAndPepper, kth_nonzero, count_nonzero, dice_coeff, hausdorff,
                        surface_metrics, pack_mask_bits, encode_flaprec_bits, RandomAffine, affine_masks,
                        RandomCraniectomy)
from . import preprocess  # noqa: F401
from .dropin import install, uninstall, MODEL_CLASSES, HANDLER_CLASSES  # noqa: F401

__version__ = "0.1.0"
