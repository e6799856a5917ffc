"""Argument rules of TranslationInferenceBeamSearchSpeculative.generate_batches(): checked before any device work (no GPU
needed), and a refused call leaves the counters untouched."""
from __future__ import annotations

import pytest
import torch

from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative


class _NoDevice:
    """Stands in for the engine: any use of it means a device call was attempted."""

    def __getattr__(self, name):
        raise AssertionError(f"device call before the argument checks ({name})")


def _gen(smart=False):
    return TranslationInferenceBeamSearchSpeculative(_NoDevice(), 100, 5, 10, 10, 288, smart, 0, 1, 2, 3)


def _counters(g):
    return (g.model_calls_num, g.accepted_tokens_num, g.produced_non_pad_tokens, g.n_drafts, g.trace)


@pytest.mark.parametrize("smart", [False, True])
def test_empty_list_returns_empty_list(smart):
    assert _gen(smart).generate_batches([]) == []


def test_slots_below_the_largest_batch_raise():
    with pytest.raises(ValueError, match="slots"):
        _gen().generate_batches([torch.ones(4, 8, dtype=torch.long), torch.ones(7, 9, dtype=torch.long)], slots=6)


def test_mixed_devices_raise():
    a = torch.ones(2, 8, dtype=torch.long)
    b = torch.ones(2, 8, dtype=torch.long, device="meta")
    with pytest.raises(ValueError, match="same device"):
        _gen().generate_batches([a, b])


@pytest.mark.parametrize("shape", [(0, 8), (3, 1), (5,)])
def test_malformed_batches_raise(shape):
    with pytest.raises(ValueError, match="batch"):
        _gen().generate_batches([torch.ones(2, 8, dtype=torch.long), torch.ones(*shape, dtype=torch.long)])


def test_smart_mode_short_source_raises_like_generate():
    # a library of Ls - 5 windows is empty: generate() raises AssertionError for such a batch (C ABI argument assert)
    with pytest.raises(AssertionError, match="number of drafts"):
        _gen(True).generate_batches([torch.ones(2, 8, dtype=torch.long), torch.ones(3, 5, dtype=torch.long)])


def test_counters_untouched_by_a_refused_call():
    for g, args in ((_gen(), dict(slots=3)), (_gen(True), {})):
        with pytest.raises((ValueError, AssertionError)):
            g.generate_batches([torch.ones(4, 5, dtype=torch.long)], **args)
        assert _counters(g) == (0, 0, 0, 0, [])
