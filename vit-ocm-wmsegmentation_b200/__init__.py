"""vit-ocm-wmsegmentation_b200: B200-native (sm_100a) drop-in for the attention-map /
sliding-window segmentation hot path of linum-uqam/ViT-OCM-WMSegmentation.

The directory name carries hyphens (it mirrors the reference repository's name); import it
through the ``vitocm_b200`` shim at the repository root:

    import vitocm_b200 as vob
    model = vob.vits.vit_small(patch_size=8, num_classes=0).cuda()
    feat, attentions, qkv = model.get_intermediate_feat(x, n=1)

Modules mirror the reference's file names: ``vision_transformer`` (SSS/dino/vision_transformer.py),
``utils`` (SSS/utils.py), ``sw_processing`` (SSS/sw_processing.py), ``model`` (SSS/model.py), ``optimizer``
(SSS/optimizer.py), ``lr_scheduler`` (SSS/lr_scheduler.py), ``pgt`` (the mask-generation loop of SSS/PGT.py).
All compute is in ``libvitocm.so`` (csrc/, C ABI in include/vitocm.h); build it with
``python vit-ocm-wmsegmentation_b200/build.py``.  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from . import vision_transformer as vits  # noqa: F401
from . import utils, sw_processing, model, optimizer, lr_scheduler, synthetic, pgt  # noqa: F401
from .vision_transformer import VisionTransformer, vit_tiny, vit_small, vit_base, LazyAttention, LazyTensor  # noqa: F401
from .utils import compute_attention, attention_masks, cropped_attention_masks, head_mean_maps, concat_crops_overlap  # noqa: F401
from ._lib import VitocmError  # noqa: F401
from .sw_processing import MosaicSegmenter, sliding_window, grid_size, mosaic_grid, shard_range, shared_pinned_u8  # noqa: F401
from .model import VisionTransformerForSimMIM, MIM, MaskGenerator, build_model  # noqa: F401

__version__ = "0.1.0"
