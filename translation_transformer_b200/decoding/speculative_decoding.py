"""Speculative decoding strategies with the reference's constructor / `generate` interface.

Reference: /root/reference/src/decoding/speculative_decoding.py.  `generate(src)` hands the whole
decoding loop to libttb200: the encoder, draft construction, KV-cached decoder steps, draft
verification, token append, retirement of finished queries and the stop test all run on the
GPU without a host round-trip per step; the host only polls a completion word.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Sequence

import torch

from .. import _lib
from ..model import B200Transformer

# generate_batches(): default query slots per query of the largest batch.  Greedy bench workload (bs 32, trained-like
# weights, 24 batches) on one B200 at 1000 W: 1908 SMILES/s one batch at a time; 1964 / 3221 / 3681 / 4151 / 4378 with
# 32 / 48 / 64 / 96 / 128 slots (profiles/r3_continuous_copy.json, DESIGN.md section 10)
DEFAULT_SLOTS_PER_BATCH = 4
# TranslationInferenceBeamSearchSpeculative.generate_batches(): default query slots per query of the largest batch (each
# slot holds n_best candidate rows), chosen from the sweep in DESIGN.md section 11
DEFAULT_BEAM_SLOTS_PER_BATCH = 16
# messages of the reference failures a batch of generate_batches() can end with (as raised by generate())
_REF_ERRORS = {
    _lib.ERR_REF_INDEX: "index out of bounds while splicing drafts into the token matrix (reference scatter, speculative_decoding.py:111)",
    _lib.ERR_REF_SHAPE: "shape mismatch: a finished row is wider than max_len (reference speculative_decoding.py:158)",
}
_BEAM_REF_ERRORS = {
    _lib.ERR_REF_SHAPE: (RuntimeError, "PAD predicted inside a hypothesis: draft slots are not contiguous (the reference fails on the "
                                       "reshape at speculative_decoding.py:524-526)"),
    _lib.ERR_REF_ASSERT: (AssertionError, "fewer candidate continuations than n_best (reference assert in topk_in_each_group, "
                                          "speculative_decoding.py:195)"),
}


def _check_batches(batches: list, slots: int | None, per_batch: int, min_len: int = 2) -> int:
    """Argument rules of generate_batches(), checked before any device work; returns the slot count.  `min_len`: the
    shortest source width the decoder's generate() accepts."""
    for b in batches:
        if b.dim() != 2 or b.shape[0] < 1 or b.shape[1] < min_len:
            raise ValueError(f"every batch must be a (B >= 1, Ls >= {min_len}) tensor of token ids, got shape {tuple(b.shape)}")
    if len({b.device for b in batches}) != 1:
        raise ValueError("all batches must be on the same device")
    bmax = max(int(b.shape[0]) for b in batches)
    if slots is None:
        slots = per_batch * bmax
    if slots < bmax:
        raise ValueError(f"slots ({slots}) must be at least the largest batch size ({bmax})")
    return slots


def _run_batches(dec, fn: str, batches: list, slots: int, params: tuple, per_query: int, traces: tuple = (),
                 widths: bool = False) -> tuple:
    """The call of library entry point `fn` common to the generate_batches() methods of decoder `dec`: device copies of the
    sources, int64 outputs of `per_query` elements per query, `params` (the loop's arguments behind the slot count),
    per-batch pointer arrays of the outputs, of the widths when `widths`, and of every entry of `traces` (a list of
    tensors, or None); then the accounting of the call's totals.  Returns (per-batch stats, widths or None, outputs)."""
    m = dec.model
    n = len(batches)
    srcs = [b.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous() for b in batches]
    outs = [torch.empty(s.shape[0] * per_query, dtype=torch.int64, device=m.device) for s in srcs]
    ptrs = lambda ts: None if ts is None else (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    sizes = (C.c_int32 * n)(*[s.shape[0] for s in srcs])
    lens = (C.c_int32 * n)(*[s.shape[1] for s in srcs])
    out_widths = (C.c_int32 * n)() if widths else None
    stats = (_lib.GenerateStats * n)()
    total = _lib.GenerateStats()
    with torch.cuda.device(m.device):
        rc = getattr(m.lib, fn)(m._h, n, ptrs(srcs), sizes, lens, slots, *params, ptrs(outs), *([out_widths] if widths else []),
                                *[ptrs(t) for t in traces], stats, C.byref(total), torch.cuda.current_stream(m.device).cuda_stream)
    _lib.check(rc, fn)
    dec.last_stats = total
    dec.gpu_launches += total.gpu_launches
    dec.gpu_ms += total.gpu_ms
    return stats, out_widths, outs


class TranslationInferenceGreedySpeculative:
    """Mirror of speculative_decoding.py:8-174 (same arguments, same counters, same output)."""

    def __init__(self, model: B200Transformer, max_len: int, draft_len: int, n_drafts: int,
                 pad_token: int, bos_token: int, eos_token: int, replace_token: int,
                 tie_break: str = "torch_cpu", keep_trace: bool = False) -> None:
        self.model = model
        self.max_len = max_len
        self.pad_token, self.bos_token, self.eos_token = pad_token, bos_token, eos_token
        self.replace_token = replace_token
        self.draft_len = draft_len
        self.n_drafts = n_drafts
        self.accepted_tokens_num = 0
        self.produced_tokens_num = 0
        self.model_calls_num = 0
        self.gpu_launches = 0
        self.gpu_ms = 0.0
        self.tie_break = {"torch_cpu": 0, "lowest_index": 1}[tie_break]
        self.keep_trace = keep_trace
        self.trace = []
        self.last_stats = None

    def __str__(self):
        return f"Greedy speculative decoding (draft_len={self.draft_len}, n_drafts={self.n_drafts}, max_len={self.max_len})"

    def generate(self, src: torch.Tensor) -> torch.Tensor:
        """(B, Ls) source token ids -> (B, 1, max_len) predictions, PAD-filled; a query that did not
        reach EOS within the width limit comes back as an all-PAD row, like in the reference."""
        m = self.model
        src_d = src.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        B, Ls = src_d.shape
        out = torch.empty(B, self.max_len, dtype=torch.int64, device=m.device)
        trace = None
        if self.keep_trace:
            trace = torch.full((self.max_len + 1, B, 4), -1, dtype=torch.int32, device=m.device)
        stats = _lib.GenerateStats()
        with torch.cuda.device(m.device):
            rc = m.lib.ttb_greedy_speculative_generate(
                m._h, src_d.data_ptr(), B, Ls, self.max_len, self.draft_len, self.n_drafts, self.pad_token,
                self.bos_token, self.eos_token, self.replace_token, self.tie_break, out.data_ptr(),
                trace.data_ptr() if trace is not None else None, C.byref(stats),
                torch.cuda.current_stream(m.device).cuda_stream)
        self.last_stats = stats
        self.model_calls_num += stats.model_calls
        self.accepted_tokens_num += stats.accepted_tokens
        self.produced_tokens_num += stats.produced_tokens
        self.gpu_launches += stats.gpu_launches
        self.gpu_ms += stats.gpu_ms
        if trace is not None:
            self._append_trace(trace, stats.model_calls)
        _lib.check(rc, "ttb_greedy_speculative_generate")
        out = out.unsqueeze(1)
        return out if src.is_cuda else out.to(src.device)

    def generate_batches(self, batches: Sequence[torch.Tensor], slots: int | None = None,
                         on_error: Callable[[int, Exception], object] | None = None) -> list:
        """Continuous batching: decode `batches` in ONE device loop whose `slots` query slots are refilled with the
        queries of the next batch as soon as enough of them are free (batches are admitted in list order).

        Returns `[self.generate(b) for b in batches]` bit for bit, and advances the counters and `trace` exactly as those
        calls would: a batch keeps the width, stop and error rules of its own batch in the shared loop.  A reference
        failure of batch i raises its RuntimeError when position i is reached, unless `on_error(i, exc)` is given,
        whose return value then stands in for that batch's result (the contract of `InFlightDecoder.map`).
        `slots` defaults to DEFAULT_SLOTS_PER_BATCH times the largest batch size."""
        batches = list(batches)
        if not batches:
            return []
        slots = _check_batches(batches, slots, DEFAULT_SLOTS_PER_BATCH)
        traces = None
        if self.keep_trace:
            traces = [torch.full((self.max_len + 1, b.shape[0], 4), -1, dtype=torch.int32, device=self.model.device) for b in batches]
        stats, _, outs = _run_batches(
            self, "ttb_greedy_speculative_generate_batches", batches, slots,
            (self.max_len, self.draft_len, self.n_drafts, self.pad_token, self.bos_token, self.eos_token, self.replace_token, self.tie_break),
            self.max_len, (traces,))
        results = []
        for i in range(len(batches)):
            st = stats[i]
            self.model_calls_num += st.model_calls
            self.accepted_tokens_num += st.accepted_tokens
            self.produced_tokens_num += st.produced_tokens
            if traces is not None:
                self._append_trace(traces[i], st.model_calls)
            if st.error:
                exc = RuntimeError(_REF_ERRORS[st.error])
                if on_error is None:
                    raise exc
                results.append(on_error(i, exc))
                continue
            out = outs[i].view(-1, 1, self.max_len)
            results.append(out if batches[i].is_cuda else out.to(batches[i].device))
        return results

    def _append_trace(self, trace: torch.Tensor, model_calls: int) -> None:
        t = trace[:model_calls].cpu()
        for it in range(t.shape[0]):
            rows = t[it][t[it, :, 0] >= 0]
            self.trace.append({"rows": rows[:, 0].tolist(), "n_accepted": rows[:, 1].tolist(),
                               "draft_index": rows[:, 2].tolist(), "width": int(rows[0, 3]) if len(rows) else 0})


class TranslationInferenceBeamSearchSpeculative:
    """Mirror of speculative_decoding.py:241-845, both draft modes (`smart_drafts_mode=False`: every candidate tries
    the n_drafts source windows, :428-598; `True`: windows of a draft library keyed by the candidate's last token,
    :600-845).  Same constructor
    arguments and counters (`model_calls_num`, `accepted_tokens_num`, `produced_non_pad_tokens`);
    `generate(src)` returns the (B, n_best, width) hypotheses best-first, like the reference."""

    def __init__(self, model: B200Transformer, max_len: int, n_best: int, draft_len: int, n_drafts: int,
                 vocab_size: int, smart_drafts_mode: bool, pad_token: int, bos_token: int, eos_token: int,
                 C_token: int, tie_break: str = "torch_cpu", keep_trace: bool = False) -> None:
        self.smart_drafts_mode = bool(smart_drafts_mode)
        self.model = model
        self.max_len = max_len
        self.vocab_size = vocab_size
        self.pad_token_idx, self.bos_token_idx, self.eos_token_idx, self.C_token_idx = pad_token, bos_token, eos_token, C_token
        self.n_best = n_best
        self.accepted_tokens_num = 0
        self.model_calls_num = 0
        self.produced_non_pad_tokens = 0
        self.requested_drafts_num = n_drafts
        self.max_draft_len, self.min_draft_len = 200, 5
        drafts_len = min(max(self.min_draft_len, draft_len), self.max_draft_len)
        if drafts_len != draft_len:
            print(f"The draft length should be in range [{self.min_draft_len}: {self.max_draft_len}], so it was changed to {drafts_len}")
        self.draft_len = drafts_len
        self.n_drafts = 0
        self.gpu_launches = 0
        self.gpu_ms = 0.0
        self.tie_break = {"torch_cpu": 0, "lowest_index": 1}[tie_break]
        self.keep_trace = keep_trace
        self.trace = []
        self.last_stats = None

    def __str__(self):
        return (f"SpeculativeSampling decoding (n_best={self.n_best}, max_len={self.max_len}, "
                f"max_num_of_drafts={self.requested_drafts_num}, draft_len={self.draft_len})")

    def generate(self, src: torch.Tensor) -> torch.Tensor:
        m = self.model
        src_d = src.to(device=m.device, dtype=torch.int64, non_blocking=True).contiguous()
        B, Ls = src_d.shape
        K, N = self.n_best, self.requested_drafts_num
        cap = self.max_len + self.draft_len + 4
        out = torch.empty(B * K * cap, dtype=torch.int64, device=m.device)
        t_nacc = t_pick = None
        if self.keep_trace:
            t_nacc = torch.full((self.max_len, B * K, N), -1, dtype=torch.int32, device=m.device)
            t_pick = torch.full((self.max_len, B * K), -1, dtype=torch.int32, device=m.device)
        stats = _lib.GenerateStats()
        width = C.c_int32(0)
        with torch.cuda.device(m.device):
            rc = m.lib.ttb_beam_speculative_generate(
                m._h, src_d.data_ptr(), B, Ls, self.max_len, K, self.draft_len, N, int(self.smart_drafts_mode), self.pad_token_idx, self.bos_token_idx,
                self.eos_token_idx, self.C_token_idx, self.tie_break, out.data_ptr(), C.byref(width),
                t_nacc.data_ptr() if t_nacc is not None else None, t_pick.data_ptr() if t_pick is not None else None,
                C.byref(stats), torch.cuda.current_stream(m.device).cuda_stream)
        self.last_stats = stats
        self.n_drafts += B * N
        self.model_calls_num += stats.model_calls
        self.accepted_tokens_num += stats.accepted_tokens
        self.produced_non_pad_tokens += stats.produced_tokens
        self.gpu_launches += stats.gpu_launches
        self.gpu_ms += stats.gpu_ms
        if t_nacc is not None:
            self._append_trace(t_nacc, t_pick, stats.model_calls)
        _lib.check(rc, "ttb_beam_speculative_generate")
        W = width.value
        res = out[:B * K * W].view(B, K, W)
        return res if src.is_cuda else res.to(src.device)

    def generate_batches(self, batches: Sequence[torch.Tensor], slots: int | None = None,
                         on_error: Callable[[int, Exception], object] | None = None) -> list:
        """Continuous batching: decode `batches` in ONE device loop whose `slots` query slots (n_best candidate rows each)
        are refilled with the queries of the next batch as soon as enough of them are free (batches are admitted whole, in
        list order, between two iterations).

        Returns `[self.generate(b) for b in batches]` bit for bit, each (B_i, n_best, W_i), and advances the counters and
        `trace` exactly as those calls would: a batch keeps the width, draft length, stop and error rules of its own batch
        in the shared loop.  A reference failure of batch i raises the exception generate() raises for it when position i
        is reached, unless `on_error(i, exc)` is given, whose return value then stands in for that batch's result.
        `slots` defaults to DEFAULT_BEAM_SLOTS_PER_BATCH times the largest batch size."""
        batches = list(batches)
        if not batches:
            return []
        slots = _check_batches(batches, slots, DEFAULT_BEAM_SLOTS_PER_BATCH)
        if self.smart_drafts_mode:
            for b in batches:
                if b.shape[1] <= 5:   # a library of Ls - 5 windows: generate() fails on such a batch as well
                    raise AssertionError("The number of drafts must be greater than 0")
        K, N = self.n_best, self.requested_drafts_num
        t_nacc = t_pick = None
        if self.keep_trace:
            t_nacc = [torch.full((self.max_len, b.shape[0] * K, N), -1, dtype=torch.int32, device=self.model.device) for b in batches]
            t_pick = [torch.full((self.max_len, b.shape[0] * K), -1, dtype=torch.int32, device=self.model.device) for b in batches]
        stats, widths, outs = _run_batches(
            self, "ttb_beam_speculative_generate_batches", batches, slots,
            (self.max_len, K, self.draft_len, N, int(self.smart_drafts_mode), self.pad_token_idx, self.bos_token_idx, self.eos_token_idx,
             self.C_token_idx, self.tie_break),
            K * (self.max_len + self.draft_len + 4), (t_nacc, t_pick), widths=True)
        results = []
        for i in range(len(batches)):
            st, B = stats[i], batches[i].shape[0]
            self.n_drafts += B * N
            self.model_calls_num += st.model_calls
            self.accepted_tokens_num += st.accepted_tokens
            self.produced_non_pad_tokens += st.produced_tokens
            if t_nacc is not None:
                self._append_trace(t_nacc[i], t_pick[i], st.model_calls)
            if st.error:
                kind, msg = _BEAM_REF_ERRORS[st.error]
                exc = kind(msg)
                if on_error is None:
                    raise exc
                results.append(on_error(i, exc))
                continue
            W = widths[i]
            res = outs[i][:B * K * W].view(B, K, W)
            results.append(res if batches[i].is_cuda else res.to(batches[i].device))
        return results

    def _append_trace(self, t_nacc: torch.Tensor, t_pick: torch.Tensor, model_calls: int) -> None:
        na, pk = t_nacc[:model_calls].cpu(), t_pick[:model_calls].cpu()
        for it in range(na.shape[0]):
            live = pk[it] >= 0
            self.trace.append({"n_accepted": na[it][live].numpy().astype("int64"), "pick": pk[it][live].numpy().astype("int64")})
