"""comet_pose_estimation_b200 -- B200-native (sm_100a) tracking hot path of COMET.

Python mirror of the reference interface for the path (SURVEY.md section 8b):

* :mod:`.blocks`  -- ``CorrBlock``, ``EfficientCorrBlock``  (comet/models/track_modules/blocks.py:351-484)
* :mod:`.utils`   -- ``bilinear_sampler``, ``sample_features4d``, ``get_2d_embedding``,
  ``get_2d_sincos_pos_embed`` (+ ``_from_grid``), ``get_1d_sincos_pos_embed`` (+ ``_from_grid``)
  (comet/models/utils.py:37-101, :724-974)
* :mod:`.track_tokens` -- the fused token assembly of ``BaseTrackerPredictor.forward``
  (comet/models/track_modules/base_track_predictor.py:153-224)
* :mod:`.base_track_predictor` -- drop-in ``BaseTrackerPredictor`` (same signature / state-dict keys) whose loop
  runs one fused kernel per iteration; :mod:`.update_former` is the torch plumbing it drives between iterations
* :mod:`.refine_track` -- drop-in ``refine_track`` / ``compute_score_fn`` / ``ShallowEncoder`` (comet/models/refine_track.py,
  blocks.py:114-196): the fine tracker's caller, feeding the kernels channels-last patch features without a copy

All arithmetic runs in hand-written CUDA kernels behind the C ABI of ``include/comet_b200.h``
(``libcomet_b200.so``).  PyTorch is used for device memory, streams and ``torch.distributed`` only.
There is no CPU fallback.
"""
from . import _lib  # noqa: F401  (fails loudly when the kernels are not built)
from .blocks import CorrBlock, EfficientCorrBlock, Upsampled2x  # noqa: F401
from .utils import (  # noqa: F401
    bilinear_sampler,
    sample_features4d,
    get_2d_embedding,
    get_2d_sincos_pos_embed,
    get_2d_sincos_pos_embed_from_grid,
    get_1d_sincos_pos_embed,
    get_1d_sincos_pos_embed_from_grid,
    upsample_bilinear_align_corners,
    instance_norm,
)
from .track_tokens import TrackTokenizer, sampled_pos_emb, transformer_dim  # noqa: F401
from .update_former import EfficientUpdateFormer  # noqa: F401
from .base_track_predictor import BaseTrackerPredictor  # noqa: F401
from .packed_frames import PackedFrames  # noqa: F401
from .refine_track import ShallowEncoder, compute_score_fn, extract_patches, inverted_score, refine_track  # noqa: F401
from .track_predictor import BasicEncoder, TrackerPredictor, split_batch  # noqa: F401

__version__ = "0.1.0"
