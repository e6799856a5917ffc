"""Teacher-forced scoring of given target sequences: how likely the model finds each candidate translation of a source.

Uses: log-likelihood and perplexity of the gold targets of a test set (`scripts/score.py`), re-ranking an n-best list
(the `(B, n_best, W)` output of the beam searches can be passed unchanged), round-trip checks of retrosynthesis
predictions with a forward model.  The whole computation runs in libttb200 (`ttb_score_targets`, DESIGN.md section 14):
the encoder and the cross-attention K/V once per source, one decoder pass over every candidate position, the vocabulary
projection reduced to the log-probability of the next target token without materialising the logits.
"""
from __future__ import annotations

from typing import NamedTuple

import torch

from . import _lib

MAX_ROWS_PER_SOURCE = 32768   # K * Lt: the decoder rows of one source must fit one chunk of the device computation


class Scores(NamedTuple):
    logp: torch.Tensor                 # (B, K) or (B,) float32: sum of the log-probabilities of the scored positions
    n_tokens: torch.Tensor             # same shape, int32: scored positions (0 when column 1 is PAD)
    token_logp: torch.Tensor | None    # (B, K, Lt - 1) or (B, Lt - 1) float32, 0 at unscored positions; only when asked


class TranslationScorer:
    """Log-likelihood of given targets under a `B200Transformer`.

    A candidate is `tgt[..., 1:]` (column 0 is the decoder's start token, given and not scored) up to and including its
    first `eos_token`, or up to but not including its first `pad_token`, whichever comes first; tokens behind that end are
    never read into the result.  Position t scores `log_softmax(decoder(src, tgt[..., :t]))[t - 1, tgt[..., t]]`, the
    reference model's teacher-forced next-token distribution.  Length-normalised ranking is `logp / n_tokens`."""

    def __init__(self, model, pad_token: int, eos_token: int) -> None:
        if pad_token == eos_token:
            raise ValueError("pad_token and eos_token must be different")
        self.model = model
        self.pad_token, self.eos_token = pad_token, eos_token

    def _check(self, src: torch.Tensor, tgt: torch.Tensor):
        m = self.model
        if src.dim() != 2:
            raise ValueError(f"src must be (B, Ls), got shape {tuple(src.shape)}")
        if tgt.dim() not in (2, 3):
            raise ValueError(f"tgt must be (B, Lt) or (B, K, Lt), got shape {tuple(tgt.shape)}")
        if src.device != tgt.device:
            raise ValueError(f"src and tgt must be on the same device ({src.device} vs {tgt.device})")
        tgt3 = tgt if tgt.dim() == 3 else tgt.unsqueeze(1)
        B, K, Lt = tgt3.shape
        if src.shape[0] != B:
            raise ValueError(f"src and tgt have different batch sizes ({src.shape[0]} vs {B})")
        if B == 0 or K == 0 or src.shape[1] == 0:
            raise ValueError("empty batch: B, K and Ls must be at least 1")
        if Lt < 2:
            raise ValueError("tgt needs a start column and at least one column to score (Lt >= 2)")
        if src.shape[1] > m.MAX_POSITIONS or Lt > m.MAX_POSITIONS:
            raise ValueError(f"sequences are limited to {m.MAX_POSITIONS} positions")
        if K * Lt > MAX_ROWS_PER_SOURCE:
            raise ValueError(f"K * Lt = {K * Lt} above {MAX_ROWS_PER_SOURCE} decoder rows per source")
        if src.dtype.is_floating_point or tgt.dtype.is_floating_point or src.dtype == torch.bool or tgt.dtype == torch.bool:
            raise ValueError("token ids must be integer tensors")
        # every value check in one device-to-host copy.  Out-of-range ids would index the embedding tables out of bounds
        # on the device; an all-PAD source row or a PAD start column leaves an attention row without a key.
        lo_s, hi_s, lo_t, hi_t, pad_src, pad_start = torch.stack([
            v.long() for v in (*torch.aminmax(src), *torch.aminmax(tgt3), (src == m.src_pad_token_i).all(dim=1).any(),
                               (tgt3[:, :, 0] == m.tgt_pad_token_i).any())]).tolist()
        for name, lo, hi, vocab in (("src", lo_s, hi_s, m.src_vocab_size), ("tgt", lo_t, hi_t, m.tgt_vocab_size)):
            if lo < 0 or hi >= vocab:
                raise ValueError(f"{name} token ids must lie in [0, {vocab}), got [{lo}, {hi}]")
        if pad_src:
            raise ValueError("a source row is all padding (its attention has no key)")
        if pad_start:
            raise ValueError("column 0 of a target (the start token) is padding (its self-attention has no key)")
        return tgt3

    def score(self, src: torch.Tensor, tgt: torch.Tensor, per_token: bool = False) -> Scores:
        """src (B, Ls) and tgt (B, K, Lt) or (B, Lt) int64 token ids, right-padded like the input and output of
        `generate()`.  Returns `Scores(logp, n_tokens, token_logp)` on src's device, shaped like tgt without its last
        dimension; `token_logp` only with `per_token=True`."""
        tgt3 = self._check(src, tgt)
        m = self.model
        B, K, Lt = tgt3.shape
        src_d = src.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        tgt_d = tgt3.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        logp = torch.empty(B, K, dtype=torch.float32, device=m.device)
        ntok = torch.empty(B, K, dtype=torch.int32, device=m.device)
        tok = torch.empty(B, K, Lt - 1, dtype=torch.float32, device=m.device) if per_token else None
        with torch.cuda.device(m.device):
            rc = m.lib.ttb_score_targets(m._h, src_d.data_ptr(), B, src_d.shape[1], tgt_d.data_ptr(), K, Lt, self.pad_token,
                                         self.eos_token, logp.data_ptr(), ntok.data_ptr(), tok.data_ptr() if per_token else None,
                                         torch.cuda.current_stream(m.device).cuda_stream)
        _lib.check(rc, "ttb_score_targets")
        if tgt.dim() == 2:
            logp, ntok, tok = logp[:, 0], ntok[:, 0], tok[:, 0] if per_token else None
        if not src.is_cuda:
            logp, ntok, tok = logp.to(src.device), ntok.to(src.device), tok.to(src.device) if per_token else None
        return Scores(logp, ntok, tok)
