"""translation_transformer_b200 — B200-native inference hot path of the Molecular Transformer.

Scope (DESIGN.md §0): the encoder/decoder forward pass driven by the speculative greedy and
beam-search decoding loops of Academich/translation-transformer, behind that project's own
`encode_src` / `decode_tgt` / `make_drafts` / `generate` / `predict_step` interface.  All device
work is done by hand-written sm_100a CUDA kernels in `csrc/` reached through the C ABI declared
in `include/ttb200.h`; PyTorch only owns device memory and `torch.distributed`.  There is no
CPU fallback: importing the package works anywhere, using it without the CUDA library raises.
"""
from .weights import ModelConfig, random_init_state_dict, infer_config, PRODUCT_PREDICTION, SINGLE_STEP_RETRO  # noqa: F401
from .scoring import Scores, TranslationScorer  # noqa: F401

__version__ = "0.1.0"
