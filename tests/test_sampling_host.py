"""Sampling decoding on the CPU: the oracle's noise generator against the Random123 known answers, the per-source key,
greedy equivalence of top_k = 1, and the argument rules of TranslationInferenceSampling.generate(), which are checked
before any device work (no GPU needed)."""
from __future__ import annotations

import math

import pytest
import torch

from helpers import SMALL
from oracle.sampling import TranslationInferenceSampling as SamplingOracle
from oracle.sampling import philox4x32_10, source_key
from oracle.standard_decoding import GreedyOracle
from oracle.transformer import OracleTransformer
from translation_transformer_b200.decoding import TranslationInferenceSampling
from translation_transformer_b200.weights import ModelConfig, random_init_state_dict

PAD, BOS, EOS, V = 0, 1, 2, 40

# Random123 known-answer vectors of Philox4x32-10: (counter, key) -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize("i", range(len(KAT)))
def test_philox_known_answers(i):
    ctr, key, want = KAT[i]
    assert tuple(int(x) for x in philox4x32_10(ctr, key)) == want


def test_key_ignores_trailing_pad():
    row = [BOS, 7, 9, 11, EOS]
    k = source_key(row, 123, PAD)
    assert source_key(row + [PAD] * 3, 123, PAD) == k
    assert source_key(row + [PAD] * 17, 123, PAD) == k
    assert source_key(row, 124, PAD) != k
    assert source_key(row[:-1], 123, PAD) != k


def test_key_is_fnv1a64_of_seed_and_tokens():
    # FNV-1a-64 of the empty string is the offset basis; one zero byte: (basis ^ 0) * prime
    basis, prime = 0xcbf29ce484222325, 0x100000001b3
    h = basis
    for byte in (5).to_bytes(8, "little") + (300).to_bytes(4, "little"):
        h = ((h ^ byte) * prime) % 2 ** 64
    assert source_key([300, PAD], 5, PAD) == h


def _model(gemm_dtype="fp32", eos_bias=0.9):
    cfg = ModelConfig(src_vocab_size=V, tgt_vocab_size=V, **SMALL)
    sd = {k: v.clone() for k, v in random_init_state_dict(cfg, 3).items()}
    sd["next_token_classifier.bias"][EOS] += eos_bias
    sd["next_token_classifier.bias"][PAD] -= 5.0
    return OracleTransformer(sd, cfg.num_heads, gemm_dtype=gemm_dtype)


def _src(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(3, V, (B, 9), generator=g)
    src[:, 0] = BOS
    src[0, 7:] = PAD
    return src


@pytest.mark.parametrize("temperature", [1.0, 0.3, 5.0])
def test_top_k_1_is_greedy_up_to_the_first_eos(temperature):
    m = _model()
    src = _src(3)
    L = 12
    greedy = GreedyOracle(m, L, PAD, BOS, EOS).generate(src)[:, 0]
    out = SamplingOracle(m, L, 4, PAD, BOS, EOS, temperature=temperature, top_k=1, seed=9).generate(src)
    for b in range(3):
        g = greedy[b]
        end = next((i for i in range(1, L) if int(g[i]) in (EOS, PAD)), L - 1)
        for s in range(4):
            assert torch.equal(out[b, s, :end + 1], g[:end + 1])
            assert bool((out[b, s, end + 1:] == PAD).all())


def test_rows_end_individually_and_counters():
    m = _model(eos_bias=2.5)
    src = _src(2)
    o = SamplingOracle(m, 10, 3, PAD, BOS, EOS, temperature=1.0, top_k=0, seed=4)
    out = o.generate(src)
    lengths = []
    drawn = 0
    for row in out.view(-1, 10):
        ends = [i for i in range(1, 10) if int(row[i]) in (EOS, PAD)]
        n = ends[0] if ends else 9
        lengths.append(n)
        drawn += n
        assert bool((row[n + 1:] == PAD).all())
    assert len(set(lengths)) > 1, "the EOS bias should end rows at different steps"
    assert o.sampled_tokens == drawn
    assert o.model_calls_num == max(lengths)
    assert o.given_tokens == int((src != PAD).sum())


def test_same_call_twice_and_seed_argument():
    m = _model()
    src = _src(2)
    o = SamplingOracle(m, 8, 3, PAD, BOS, EOS, temperature=0.8, top_k=5, seed=1)
    a, b = o.generate(src), o.generate(src)
    assert torch.equal(a, b)
    assert torch.equal(o.generate(src, seed=1), a)
    assert not torch.equal(o.generate(src, seed=2), a)


class _Stand:
    """Stands in for the engine: the shape attributes a caller reads, and any other use means a device call was attempted."""
    src_vocab_size = tgt_vocab_size = V
    src_pad_token_i = tgt_pad_token_i = PAD
    MAX_POSITIONS = 1024

    def __getattr__(self, name):
        raise AssertionError(f"device call before the argument checks ({name})")


OK = dict(max_len=10, n_samples=3, pad_token=PAD, bos_token=BOS, eos_token=EOS, temperature=1.0, top_k=0, seed=0)

BAD = {
    "src_1d": ({}, lambda: _src(2)[0], "src"),
    "src_3d": ({}, lambda: _src(2)[:, None], "src"),
    "n_samples_0": ({"n_samples": 0}, None, "n_samples"),
    "too_many_rows": ({"n_samples": 1025}, None, "2048"),
    "temperature_0": ({"temperature": 0.0}, None, "temperature"),
    "temperature_negative": ({"temperature": -1.0}, None, "temperature"),
    "temperature_inf": ({"temperature": math.inf}, None, "temperature"),
    "temperature_nan": ({"temperature": math.nan}, None, "temperature"),
    "top_k_negative": ({"top_k": -1}, None, "top_k"),
    "top_k_above_vocab": ({"top_k": V + 1}, None, "top_k"),
    "max_len_1": ({"max_len": 1}, None, "max_len"),
    "pad_equals_eos": ({"eos_token": PAD}, None, "different"),
    "max_len_above_table": ({"max_len": 1023}, None, "limited"),
    "src_above_table": ({}, lambda: torch.ones(1, 1025, dtype=torch.long), "limited"),
    "seed_negative": ({"seed": -1}, None, "seed"),
    "seed_too_large": ({"seed": 2 ** 64}, None, "seed"),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_bad_arguments_raise_before_device_work(case):
    kw, make_src, match = BAD[case]
    src = make_src() if make_src else _src(2)
    with pytest.raises(ValueError, match=match):
        TranslationInferenceSampling(_Stand(), **{**OK, **kw}).generate(src)


def test_bad_seed_argument_of_generate_raises():
    with pytest.raises(ValueError, match="seed"):
        TranslationInferenceSampling(_Stand(), **OK).generate(_src(2), seed=2 ** 64)


def test_valid_arguments_reach_the_engine():
    for kw in ({}, {"top_k": V, "seed": 2 ** 64 - 1}, {"n_samples": 1024, "top_k": 1}):
        with pytest.raises(AssertionError, match="device call"):
            TranslationInferenceSampling(_Stand(), **{**OK, **kw}).generate(_src(2))
