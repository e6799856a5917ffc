"""Teacher-forced scoring on the CPU: the scored-range rule of the oracle (oracle/scoring.py) on hand cases, against
independent per-candidate runs on the truncated candidates, and the argument rules of TranslationScorer.score(), which are
checked before any device work (no GPU needed)."""
from __future__ import annotations

import pytest
import torch
import torch.nn.functional as F

from helpers import SMALL
from oracle.scoring import score as oracle_score
from oracle.transformer import OracleTransformer
from translation_transformer_b200 import TranslationScorer
from translation_transformer_b200.weights import ModelConfig, random_init_state_dict

PAD, BOS, EOS, V = 0, 1, 2, 40

# (target row, scored positions)
CASES = {
    "eos_at_1": ([BOS, EOS, 5, 6, 7, 8], 1),
    "pad_at_1": ([BOS, PAD, 5, 6, EOS, 8], 0),
    "no_eos_no_pad": ([BOS, 5, 6, 7, 8, 9], 5),
    "pad_before_eos": ([BOS, 5, 6, PAD, EOS, 9], 2),
    "tokens_after_eos": ([BOS, 5, 6, EOS, 7, 8], 3),
}


def _model(gemm_dtype):
    cfg = ModelConfig(src_vocab_size=V, tgt_vocab_size=V, **SMALL)
    return OracleTransformer(random_init_state_dict(cfg, 3), cfg.num_heads, gemm_dtype=gemm_dtype)


def _src(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(3, V, (B, 9), generator=g)
    src[:, 0] = BOS
    src[0, 7:] = PAD
    return src


@pytest.mark.parametrize("gemm_dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_scored_range_against_truncated_runs(case, gemm_dtype):
    row, n = CASES[case]
    m = _model(gemm_dtype)
    src = _src(1)
    tgt = torch.tensor(row)[None, None]
    logp, ntok, tok = oracle_score(m, src, tgt, PAD, EOS)
    assert int(ntok) == n
    assert bool((tok[0, 0, n:] == 0).all())
    # the definition: one teacher-forced run on the candidate alone (start column + its n tokens)
    cand = tgt[0, :, :n + 1]
    want = F.log_softmax(m(src, cand)[0, :-1], dim=-1).gather(-1, cand[0, 1:, None])[:, 0] if n else torch.zeros(0)
    torch.testing.assert_close(tok[0, 0, :n], want, rtol=0, atol=2e-5)
    torch.testing.assert_close(logp[0, 0], want.sum(), rtol=0, atol=2e-5 * max(n, 1))
    if n == 0:
        assert float(logp) == 0.0


@pytest.mark.parametrize("gemm_dtype", ["fp32", "bf16"])
def test_tokens_behind_the_end_do_not_change_the_result(gemm_dtype):
    m = _model(gemm_dtype)
    rows = [CASES[c][0] for c in sorted(CASES)]
    tgt = torch.tensor(rows).view(1, len(rows), -1).repeat(2, 1, 1)
    src = _src(2)
    ref = oracle_score(m, src, tgt, PAD, EOS)
    g = torch.Generator().manual_seed(5)
    changed = tgt.clone()
    n = ref[1]
    for b in range(2):
        for k in range(len(rows)):
            lo = min(int(n[b, k]) + 2, changed.shape[2])   # the column behind the end stays (a terminating PAD must stay PAD)
            changed[b, k, lo:] = torch.randint(0, V, (changed.shape[2] - lo,), generator=g)
    assert not torch.equal(changed, tgt)
    out = oracle_score(m, src, changed, PAD, EOS)
    for a, b in zip(ref, out):
        assert torch.equal(a, b)


class _Stand:
    """Stands in for the engine: the shape attributes a caller reads, and any other use means a device call was attempted."""
    src_vocab_size = tgt_vocab_size = V
    src_pad_token_i = tgt_pad_token_i = PAD
    MAX_POSITIONS = 1024

    def __getattr__(self, name):
        raise AssertionError(f"device call before the argument checks ({name})")


def _ok():
    src = _src(2)
    tgt = torch.full((2, 3, 6), PAD, dtype=torch.long)
    tgt[:, :, 0] = BOS
    tgt[:, :, 1:4] = 7
    return src, tgt


def _bad(**kw):
    src, tgt = _ok()
    return kw.get("src", src), kw.get("tgt", tgt)


def _with(t, idx, value):
    t = t.clone()
    t[idx] = value
    return t


BAD = {
    "src_1d": (lambda: _bad(src=_ok()[0][0]), "src"),
    "src_3d": (lambda: _bad(src=_ok()[0][:, None]), "src"),
    "tgt_1d": (lambda: _bad(tgt=_ok()[1][0, 0]), "tgt"),
    "tgt_4d": (lambda: _bad(tgt=_ok()[1][None]), "tgt"),
    "batch_mismatch": (lambda: _bad(tgt=_ok()[1][:1]), "batch"),
    "empty_batch": (lambda: (_ok()[0][:0], _ok()[1][:0]), "empty"),
    "no_candidates": (lambda: _bad(tgt=_ok()[1][:, :0]), "empty"),
    "lt_1": (lambda: _bad(tgt=_ok()[1][:, :, :1]), "Lt"),
    "devices": (lambda: _bad(tgt=_ok()[1].to("meta")), "same device"),
    "tgt_id_too_large": (lambda: _bad(tgt=_with(_ok()[1], (1, 2, 3), V)), "tgt token ids"),
    "tgt_id_negative": (lambda: _bad(tgt=_with(_ok()[1], (0, 0, 5), -1)), "tgt token ids"),
    "src_id_too_large": (lambda: _bad(src=_with(_ok()[0], (1, 4), V + 3)), "src token ids"),
    "all_pad_source": (lambda: _bad(src=_with(_ok()[0], (1, slice(None)), PAD)), "all padding"),
    "pad_start_column": (lambda: _bad(tgt=_with(_ok()[1], (0, 1, 0), PAD)), "start token"),
    "float_tokens": (lambda: _bad(tgt=_ok()[1].float()), "integer"),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_bad_arguments_raise_before_device_work(case):
    make, match = BAD[case]
    src, tgt = make()
    with pytest.raises(ValueError, match=match):
        TranslationScorer(_Stand(), PAD, EOS).score(src, tgt)


def test_too_many_rows_per_source_raise():
    src = _src(1)
    tgt = torch.full((1, 40, 1000), 5, dtype=torch.long)
    with pytest.raises(ValueError, match="32768"):
        TranslationScorer(_Stand(), PAD, EOS).score(src, tgt)


def test_valid_arguments_reach_the_engine():
    src, tgt = _ok()
    for t in (tgt, tgt[:, 0]):
        with pytest.raises(AssertionError, match="device call"):
            TranslationScorer(_Stand(), PAD, EOS).score(src, t)


def test_pad_equal_to_eos_raises():
    with pytest.raises(ValueError, match="different"):
        TranslationScorer(_Stand(), PAD, PAD)
