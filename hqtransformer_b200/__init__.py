"""hqtransformer_b200 - B200-native (sm_100a) engine for HQ-Transformer's hierarchical sampling loop.

Drop-in surface (names and call signatures of the reference, kakaobrain/hqtransformer):
    sampling_ihqgpt, cutoff_topk_logits, cutoff_topp_probs, get_positional_encoding   (hqvae/utils/sampling.py)
    iHQGPT(...).sampling_step                                                        (hqvae/models/stage2/hierarchical_ar.py)
    ImageGPT2(config).sample, .stage2                                                (hqvae/models/__init__.py)
    load_config (YAML with the defaults of hqvae/utils/config2.py)
    HQTransformer, sampling_hqtransformer (3-level model)                            (hqvae/models/stage2/hqtransformer.py)
    HQVAEDecoder(...).decode_code                                                    (hqvae/models/stage1/generator.py)

All compute runs in libhqgraft.so (hand-written CUDA behind the C ABI in include/hqgraft.h); importing
the package without the built library raises - there is no CPU or PyTorch fallback.
"""
from ._lib import HQError, load as _load_library

_load_library()

from .config import load_config, merge_config  # noqa: E402
from .engine import Engine, SamplingParams  # noqa: E402
from .models import ImageGPT2, iHQGPT  # noqa: E402
from .sampling import (codes_to_grids, cutoff_topk_logits, cutoff_topp_probs, encode_prompts,  # noqa: E402
                       get_positional_encoding, grids_to_codes, sampling_ihqgpt, step_logits)
from .distributed import sampling_ihqgpt_sharded, shard_range  # noqa: E402
from .stage1 import HQVAEDecoder  # noqa: E402
from .hqtransformer3 import HQTransformer, sampling_hqtransformer, step_logits3  # noqa: E402

__all__ = ["HQError", "Engine", "SamplingParams", "ImageGPT2", "iHQGPT", "load_config", "merge_config",
           "sampling_ihqgpt", "step_logits", "cutoff_topk_logits", "cutoff_topp_probs", "get_positional_encoding",
           "codes_to_grids", "grids_to_codes", "encode_prompts", "sampling_ihqgpt_sharded", "shard_range", "HQVAEDecoder", "HQTransformer", "sampling_hqtransformer", "step_logits3"]
