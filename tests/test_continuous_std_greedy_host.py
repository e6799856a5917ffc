"""Argument rules of TranslationInferenceGreedy.generate_batches(): checked before any device work (no GPU needed), and a refused
call leaves the counters untouched."""
from __future__ import annotations

import pytest
import torch

from translation_transformer_b200.decoding import TranslationInferenceGreedy


class _NoDevice:
    """Stands in for the engine: any use of it means a device call was attempted."""

    def __getattr__(self, name):
        raise AssertionError(f"device call before the argument checks ({name})")


def _gen():
    return TranslationInferenceGreedy(_NoDevice(), 100, 0, 1, 2)


def _counters(g):
    return (g.model_calls_num, g.given_tokens, g.gpu_launches, g.gpu_ms, g.last_stats)


def test_empty_list_returns_empty_list():
    assert _gen().generate_batches([]) == []


def test_slots_below_the_largest_batch_raise():
    with pytest.raises(ValueError, match="slots"):
        _gen().generate_batches([torch.ones(4, 8, dtype=torch.long), torch.ones(7, 9, dtype=torch.long)], slots=6)


def test_mixed_devices_raise():
    a = torch.ones(2, 8, dtype=torch.long)
    b = torch.ones(2, 8, dtype=torch.long, device="meta")
    with pytest.raises(ValueError, match="same device"):
        _gen().generate_batches([a, b])


@pytest.mark.parametrize("shape", [(0, 8), (3, 0), (5,), (2, 3, 4)])
def test_malformed_batches_raise(shape):
    with pytest.raises(ValueError, match="batch"):
        _gen().generate_batches([torch.ones(2, 8, dtype=torch.long), torch.ones(*shape, dtype=torch.long)])


def test_one_token_sources_pass_the_checks():
    # generate() accepts (B, 1) sources: the checks let them through, and the call reaches the engine
    with pytest.raises(AssertionError, match="device call"):
        _gen().generate_batches([torch.ones(3, 1, dtype=torch.long)])


def test_counters_untouched_by_a_refused_call():
    g = _gen()
    for batches, args in (([torch.ones(4, 5, dtype=torch.long)], dict(slots=3)), ([torch.ones(4, 5, dtype=torch.long), torch.ones(3)], {})):
        with pytest.raises(ValueError):
            g.generate_batches(batches, **args)
        assert _counters(g) == (0, 0, 0, 0.0, None)
