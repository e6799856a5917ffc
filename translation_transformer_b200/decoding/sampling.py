"""Sampling decoding: several seeded random translations per source, drawn from the model's distribution.

`TranslationInferenceSampling.generate(src)` returns (B, n_samples, max_len) token ids.  Unlike a beam search, which returns
the n most likely sequences (often near-duplicates), the samples are a diverse set drawn from softmax(logits / temperature),
optionally restricted to the top_k most likely tokens of every step (OpenNMT-py's random sampling).  Uses: candidate
generation for retrosynthesis, round-trip filtering with a forward model, estimating how uncertain the model is about a
product.  To rank or score the samples pass the output unchanged to `TranslationScorer.score(src, samples)`.

The whole loop runs in libttb200 (`ttb_sample_generate`, DESIGN.md section 15): the encoder and the cross-attention K/V
once per source, the KV-cached greedy loop over B * n_samples sample rows that end individually, and the draw fused into
the vocabulary projection (a Gumbel-max epilogue; the logits never reach memory on the bf16 path).

Reproducibility: the noise of a source comes from a counter-based generator keyed by the seed and the source's non-PAD
tokens, so a query's samples depend only on its source tokens, the seed and the settings (n_samples, temperature, top_k,
max_len, weights, precision) -- not on its position in the batch, the other queries or which engine decodes it.  Two
identical calls return the same tensor, and identical sources with the same seed get identical samples.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from .. import _lib

MAX_SAMPLE_ROWS = 2048   # B * n_samples: the slot limit of the device loops


class TranslationInferenceSampling:
    """Seeded temperature / top-k sampling.

    Sample s of source b starts from `bos_token` and appends one drawn token per step; a row ends at its first drawn
    `eos_token` or `pad_token` (kept), or when it holds `max_len` tokens, and is PAD behind.  The token at column t is
    argmax_v (logit_v / temperature + g_v) over the candidates (all tokens for top_k = 0, else the top_k largest logits),
    g_v Gumbel noise from Philox4x32-10; `top_k = 1` is greedy for any temperature.  `seed` in [0, 2^64); the seed does not
    advance between calls.  Counters: `model_calls_num` (decoder steps), `given_tokens` (non-PAD source tokens),
    `sampled_tokens` (drawn tokens), `gpu_launches`, `gpu_ms`, `last_stats` (`unfinished`: rows that reached max_len
    without EOS or PAD)."""

    def __init__(self, model, max_len: int, n_samples: int, pad_token: int, bos_token: int, eos_token: int,
                 temperature: float = 1.0, top_k: int = 0, seed: int = 0) -> None:
        self.model = model
        self.max_len, self.n_samples = max_len, n_samples
        self.pad_token, self.bos_token, self.eos_token = pad_token, bos_token, eos_token
        self.temperature, self.top_k, self.seed = temperature, top_k, seed
        self.model_calls_num = 0
        self.given_tokens = 0
        self.sampled_tokens = 0
        self.gpu_launches = 0
        self.gpu_ms = 0.0
        self.last_stats = None

    def __str__(self):
        return (f"Sampling decoding (n_samples={self.n_samples}, temperature={self.temperature}, top_k={self.top_k}, "
                f"seed={self.seed}, max_len={self.max_len})")

    def _check(self, src: torch.Tensor, seed) -> int:
        m = self.model
        if src.dim() != 2:
            raise ValueError(f"src must be (B, Ls), got shape {tuple(src.shape)}")
        B, Ls = src.shape
        if B == 0 or Ls == 0:
            raise ValueError("empty batch: B and Ls must be at least 1")
        if not isinstance(self.n_samples, int) or self.n_samples < 1:
            raise ValueError(f"n_samples must be an integer >= 1, got {self.n_samples}")
        if B * self.n_samples > MAX_SAMPLE_ROWS:
            raise ValueError(f"B * n_samples = {B * self.n_samples} above {MAX_SAMPLE_ROWS} sample rows")
        T = float(self.temperature)
        if not (math.isfinite(T) and T > 0.0):
            raise ValueError(f"temperature must be finite and > 0, got {self.temperature}")
        if not isinstance(self.top_k, int) or not 0 <= self.top_k <= m.tgt_vocab_size:
            raise ValueError(f"top_k must lie in [0, {m.tgt_vocab_size}], got {self.top_k}")
        if self.max_len < 2:
            raise ValueError(f"max_len must be at least 2, got {self.max_len}")
        if self.pad_token == self.eos_token:
            raise ValueError("pad_token and eos_token must be different")
        if Ls > m.MAX_POSITIONS or self.max_len + 2 > m.MAX_POSITIONS:
            raise ValueError(f"sequences are limited to {m.MAX_POSITIONS} source positions and {m.MAX_POSITIONS - 2} target tokens")
        seed = self.seed if seed is None else seed
        if not isinstance(seed, int) or not 0 <= seed < 2 ** 64:
            raise ValueError(f"seed must be an integer in [0, 2^64), got {seed}")
        return seed

    def generate(self, src: torch.Tensor, seed: int | None = None) -> torch.Tensor:
        """(B, Ls) source token ids -> (B, n_samples, max_len) int64 samples on src's device.  `seed=None` takes the
        constructor's seed."""
        seed = self._check(src, seed)
        m = self.model
        src_d = src.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        B, Ls = src_d.shape
        S = self.n_samples
        out = torch.empty(B, S, self.max_len, dtype=torch.int64, device=m.device)
        stats = _lib.GenerateStats()
        with torch.cuda.device(m.device):
            rc = m.lib.ttb_sample_generate(m._h, src_d.data_ptr(), B, Ls, self.max_len, S, float(self.temperature), self.top_k,
                                           seed, self.pad_token, self.bos_token, self.eos_token, out.data_ptr(), C.byref(stats),
                                           torch.cuda.current_stream(m.device).cuda_stream)
        _lib.check(rc, "ttb_sample_generate")
        self.last_stats = stats
        self.model_calls_num += stats.model_calls
        self.given_tokens += int((src_d != m.src_pad_token_i).sum().item())
        self.sampled_tokens += stats.produced_tokens
        self.gpu_launches += stats.gpu_launches
        self.gpu_ms += stats.gpu_ms
        return out if src.is_cuda else out.to(src.device)
