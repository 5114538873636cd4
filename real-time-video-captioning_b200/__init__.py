"""gitb200: B200-native (sm_100a) implementation of the GIT captioning hot path of
farazali7/real-time-video-captioning, behind the reference's own Python model interface.

    import importlib; g = importlib.import_module("real-time-video-captioning_b200")   # or: import gitb200
    teacher = g.GenerativeImageTextTeacher.from_random_init({"num_image_with_embedding": 6})
    results = teacher(frames)          # frames [B, 6, 3, 224, 224] fp32

All compute runs in libgitb200.so (include/gitb200.h); importing works without a GPU, running does not."""
from ._lib import GitB200Error, LIB_PATH  # noqa: F401
from .engine import Engine, SearchConfig, make_config, preprocess_frames, VIT_CONFIGS  # noqa: F401
from .model import (BeamHypotheses, CLIPVisionTower, GenerativeImageTextModel, GenerativeImageTextTeacher,  # noqa: F401
                    GeneratorWithBeamSearchV2, LazyLogits, MultiStreamCaptioner, StreamingCaptioner, SyntheticTokenizer, TransformerDecoderTextualHead,
                    get_git_model)
from .student import DistillationTrainer, StudentCandidateV1  # noqa: F401
from .metrics import calculate_bleu_score_corpus  # noqa: F401
from .dist import all_reduce_bucket, caption_sharded, finish_all_reduce, shard_range  # noqa: F401

__all__ = ["Engine", "SearchConfig", "GenerativeImageTextModel", "GenerativeImageTextTeacher",
           "GeneratorWithBeamSearchV2", "get_git_model", "calculate_bleu_score_corpus", "shard_range",
           "caption_sharded", "GitB200Error", "StudentCandidateV1", "DistillationTrainer", "all_reduce_bucket",
           "finish_all_reduce", "MultiStreamCaptioner"]
