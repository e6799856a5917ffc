"""Standard (non-speculative) decoding strategies with the reference's constructor / `generate` interface.

Reference: /root/reference/src/decoding/standard_decoding.py.  `TranslationInferenceGreedy.generate` hands the whole
loop to libttb200: it is the KV-cached device loop of the speculative greedy decoding run with one row per query and
no draft tokens (one CUDA-graph replay per generated token, no host round-trip per step).
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import torch

from .. import _lib
from ..model import B200Transformer
from .speculative_decoding import _check_batches, _run_batches

# TranslationInferenceBeamSearch.generate_batches(): default query slots per query of the largest batch (each slot holds
# beam_size hypotheses).  Trained-like bench batches on one B200 at 1000 W, 1 / 2 / 4 / 8 / 16 x bs slots: 145 / 262 / 473 /
# 739 / 1051 SMILES/s (bs 4, beam 5) and 281 / 462 / 676 / 897 / 1095 (retro, bs 8, beam 10), against 138 and 261 one batch
# at a time (profiles/r5_continuous_std_beam_*.json, DESIGN.md section 12)
DEFAULT_STD_BEAM_SLOTS_PER_BATCH = 16
# TranslationInferenceGreedy.generate_batches(): default query slots per query of the largest batch.  Greedy bench workload's
# model and batches (bs 32, trained-like weights, 24 batches) on one B200 at 1000 W, 1 / 2 / 4 / 8 / 16 x bs slots: 823 / 1392 /
# 2018 / 2802 / 3160 SMILES/s, against 780 one batch at a time (profiles/r6_continuous_std_greedy_copy.json, DESIGN.md section 13)
DEFAULT_GREEDY_SLOTS_PER_BATCH = 16


class TranslationInferenceGreedy:
    """Mirror of standard_decoding.py:4-56 (same arguments, counters and output)."""

    def __init__(self, model: B200Transformer, max_len: int, pad_token: int, bos_token: int, eos_token: int) -> None:
        self.model = model
        self.max_len = max_len
        self.pad_token, self.bos_token, self.eos_token = pad_token, bos_token, eos_token
        self.model_calls_num = 0
        self.given_tokens = 0
        self.gpu_launches = 0
        self.gpu_ms = 0.0
        self.last_stats = None

    def __str__(self):
        return f"Greedy decoding (max_len={self.max_len})"

    def generate(self, src: torch.Tensor) -> torch.Tensor:
        """(B, Ls) source token ids -> (B, 1, max_len) tokens.  Like the reference, decoding stops at the first step in
        which every row predicts EOS or PAD; rows that finished earlier keep their later predictions."""
        m = self.model
        src_d = src.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        B, Ls = src_d.shape
        out = torch.empty(B, self.max_len, dtype=torch.int64, device=m.device)
        stats = _lib.GenerateStats()
        with torch.cuda.device(m.device):
            rc = m.lib.ttb_greedy_generate(m._h, src_d.data_ptr(), B, Ls, self.max_len, self.pad_token, self.bos_token,
                                           self.eos_token, out.data_ptr(), C.byref(stats),
                                           torch.cuda.current_stream(m.device).cuda_stream)
        _lib.check(rc, "ttb_greedy_generate")
        self.last_stats = stats
        self.model_calls_num += stats.model_calls
        self.given_tokens += int((src_d != m.src_pad_token_i).sum().item())
        self.gpu_launches += stats.gpu_launches
        self.gpu_ms += stats.gpu_ms
        out = out.unsqueeze(1)
        return out if src.is_cuda else out.to(src.device)

    def generate_batches(self, batches: Sequence[torch.Tensor], slots: int | None = None) -> list:
        """Continuous batching: decode `batches` in ONE device loop whose `slots` query slots are refilled with the queries
        of the next batch as soon as enough of them are free (batches are admitted whole, in list order, between two steps;
        a batch frees its slots when it stops).

        Returns `[self.generate(b) for b in batches]` bit for bit, each (B_i, 1, max_len), and advances the counters as
        those calls would: a batch keeps the step count and stop rule of its own batch in the shared loop.  `slots`
        defaults to DEFAULT_GREEDY_SLOTS_PER_BATCH times the largest batch size."""
        batches = list(batches)
        if not batches:
            return []
        slots = _check_batches(batches, slots, DEFAULT_GREEDY_SLOTS_PER_BATCH, min_len=1)   # generate() takes Ls = 1 too
        stats, _, outs = _run_batches(self, "ttb_greedy_generate_batches", batches, slots,
                                      (self.max_len, self.pad_token, self.bos_token, self.eos_token), self.max_len)
        results = []
        for i in range(len(batches)):
            self.model_calls_num += stats[i].model_calls
            self.given_tokens += int((batches[i] != self.model.src_pad_token_i).sum().item())
            out = outs[i].view(-1, 1, self.max_len)
            results.append(out if batches[i].is_cuda else out.to(batches[i].device))
        return results


class TranslationInferenceBeamSearch:
    """Mirror of standard_decoding.py:59-174 (same arguments, counters and output): `generate(src)` returns the
    (B, beam_size, width) hypotheses best-first; width is the number of generated columns."""

    def __init__(self, model: B200Transformer, beam_size: int, max_len: int, pad_token: int, bos_token: int, eos_token: int):
        assert max_len > 1
        assert beam_size > 0
        self.model = model
        self.beam_size, self.max_len = beam_size, max_len
        self.pad_token, self.bos_token, self.eos_token = pad_token, bos_token, eos_token
        self.model_calls_num = 0
        self.given_tokens = 0
        self.b_sz = 0
        self.gpu_launches = 0
        self.gpu_ms = 0.0
        self.last_stats = None

    def __str__(self):
        return f"Beam search decoding (beam_size={self.beam_size}, max_len={self.max_len})"

    def generate(self, src: torch.Tensor) -> torch.Tensor:
        m = self.model
        src_d = src.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        B, Ls = src_d.shape
        out = torch.empty(B * self.beam_size * self.max_len, dtype=torch.int64, device=m.device)
        stats = _lib.GenerateStats()
        width = C.c_int32(0)
        with torch.cuda.device(m.device):
            rc = m.lib.ttb_beam_search_generate(m._h, src_d.data_ptr(), B, Ls, self.max_len, self.beam_size, self.pad_token,
                                                self.bos_token, self.eos_token, out.data_ptr(), C.byref(width), C.byref(stats),
                                                torch.cuda.current_stream(m.device).cuda_stream)
        _lib.check(rc, "ttb_beam_search_generate")
        self.last_stats = stats
        self.model_calls_num += stats.model_calls
        self.given_tokens += int((src_d != m.src_pad_token_i).sum().item())
        self.gpu_launches += stats.gpu_launches
        self.gpu_ms += stats.gpu_ms
        W = width.value
        res = out[:B * self.beam_size * W].view(B, self.beam_size, W)
        return res if src.is_cuda else res.to(src.device)

    def generate_batches(self, batches: Sequence[torch.Tensor], slots: int | None = None) -> list:
        """Continuous batching: decode `batches` in ONE device loop whose `slots` query slots (beam_size hypotheses each)
        are refilled with the queries of the next batch as soon as enough of them are free (batches are admitted whole, in
        list order, between two steps; a batch frees its slots when it stops).

        Returns `[self.generate(b) for b in batches]` bit for bit, each (B_i, beam_size, W_i), and advances the counters
        as those calls would: a batch keeps the width, first step and stop rule of its own batch in the shared loop.
        `slots` defaults to DEFAULT_STD_BEAM_SLOTS_PER_BATCH times the largest batch size."""
        batches = list(batches)
        if not batches:
            return []
        slots = _check_batches(batches, slots, DEFAULT_STD_BEAM_SLOTS_PER_BATCH, min_len=1)   # generate() takes Ls = 1 too
        K = self.beam_size
        stats, widths, outs = _run_batches(self, "ttb_beam_search_generate_batches", batches, slots,
                                           (self.max_len, K, self.pad_token, self.bos_token, self.eos_token), K * self.max_len, widths=True)
        results = []
        for i in range(len(batches)):
            B, W = batches[i].shape[0], widths[i]
            self.model_calls_num += stats[i].model_calls
            self.given_tokens += int((batches[i] != self.model.src_pad_token_i).sum().item())
            res = outs[i][:B * K * W].view(B, K, W)
            results.append(res if batches[i].is_cuda else res.to(batches[i].device))
        return results
