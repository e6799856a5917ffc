"""Oracle (test infrastructure): teacher-forced scoring of given targets on the CPU (DESIGN.md section 14).

Candidate (b, k) is tgt[b, k, 1:] up to and including its first EOS, or up to but not including its first PAD, whichever
comes first.  Position t is scored with log_softmax(forward(src[b], tgt[b, k, :t]))[t - 1, tgt[b, k, t]].  The decoder is
causal, so one forward pass over the whole row gives the teacher-forced distribution of every prefix; tokens behind a
candidate's end change neither its scored positions nor (being masked or causally invisible) their values.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .transformer import OracleTransformer


def scored_lengths(tgt: torch.Tensor, pad: int, eos: int) -> torch.Tensor:
    """(..., Lt) -> (...) int64 number of scored positions of every candidate."""
    body = tgt[..., 1:]
    Lt1 = body.shape[-1]
    idx = torch.arange(1, Lt1 + 1).expand_as(body)
    big = torch.full_like(body, Lt1 + 1)
    first_eos = torch.where(body == eos, idx, big).amin(dim=-1)       # 1-based column of the first EOS
    first_pad = torch.where(body == pad, idx, big).amin(dim=-1)
    n = torch.minimum(first_eos, first_pad - 1)
    return n.clamp(max=Lt1)


def score(model: OracleTransformer, src: torch.Tensor, tgt: torch.Tensor, pad: int, eos: int):
    """src (B, Ls), tgt (B, K, Lt) -> (logp_sum (B, K) f32, n_tokens (B, K) int32, token_logp (B, K, Lt - 1) f32)."""
    B, K, Lt = tgt.shape
    logits = model(src.repeat_interleave(K, 0), tgt.reshape(B * K, Lt))[:, :-1]       # row t - 1 predicts column t
    lp = F.log_softmax(logits, dim=-1).gather(-1, tgt.reshape(B * K, Lt)[:, 1:, None])[..., 0].reshape(B, K, Lt - 1)
    n = scored_lengths(tgt, pad, eos)
    scored = torch.arange(1, Lt)[None, None, :] <= n[..., None]
    token_logp = torch.where(scored, lp, torch.zeros(()))
    return token_logp.sum(dim=-1), n.to(torch.int32), token_logp
