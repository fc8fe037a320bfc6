"""B200-native hot path of APTP (rezashkv/diffusion_pruning): the per-sample, architecture-code-gated
SD-2.1 U-Net denoising step and its router, as hand-written sm_100a CUDA behind the reference's
`pdm.models` interface. See DESIGN.md / INTEGRATION.md."""
from .hypernet import HyperStructure
from .mixture import PrunedExpertMixture
from .quantizer import StructureVectorQuantizer, hard_concrete
from .unet import UNet2DConditionModelGated, UNet2DConditionModelPruned, UNet2DConditionOutput

__all__ = ["UNet2DConditionModelGated", "UNet2DConditionModelPruned", "UNet2DConditionOutput", "HyperStructure", "StructureVectorQuantizer",
           "hard_concrete", "PrunedExpertMixture"]
