from .speculative_decoding import TranslationInferenceBeamSearchSpeculative, TranslationInferenceGreedySpeculative  # noqa: F401
from .standard_decoding import TranslationInferenceBeamSearch, TranslationInferenceGreedy  # noqa: F401
from .sampling import TranslationInferenceSampling  # noqa: F401
