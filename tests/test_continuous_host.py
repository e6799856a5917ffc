"""Argument rules of generate_batches(): checked before any device work (no GPU needed)."""
from __future__ import annotations

import pytest
import torch

from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative


class _NoDevice:
    """Stands in for the engine: any use of it means a device call was attempted."""

    def __getattr__(self, name):
        raise AssertionError(f"device call before the argument checks ({name})")


def _gen():
    return TranslationInferenceGreedySpeculative(_NoDevice(), 200, 10, 23, 0, 1, 2, 3)


def test_empty_list_returns_empty_list():
    assert _gen().generate_batches([]) == []


def test_slots_below_the_largest_batch_raise():
    with pytest.raises(ValueError, match="slots"):
        _gen().generate_batches([torch.ones(4, 6, dtype=torch.long), torch.ones(7, 5, dtype=torch.long)], slots=6)


def test_mixed_devices_raise():
    a = torch.ones(2, 5, dtype=torch.long)
    b = torch.ones(2, 5, dtype=torch.long, device="meta")
    with pytest.raises(ValueError, match="same device"):
        _gen().generate_batches([a, b])


@pytest.mark.parametrize("shape", [(0, 5), (3, 1), (5,)])
def test_malformed_batches_raise(shape):
    with pytest.raises(ValueError, match="batch"):
        _gen().generate_batches([torch.ones(2, 5, dtype=torch.long), torch.ones(*shape, dtype=torch.long)])


def test_counters_untouched_by_a_refused_call():
    g = _gen()
    with pytest.raises(ValueError):
        g.generate_batches([torch.ones(4, 6, dtype=torch.long)], slots=3)
    assert (g.model_calls_num, g.accepted_tokens_num, g.produced_tokens_num, g.trace) == (0, 0, 0, [])
