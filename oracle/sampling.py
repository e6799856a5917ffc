"""Oracle (test infrastructure): the sampling decoding on the CPU (DESIGN.md section 15).

`TranslationInferenceSampling(model, max_len, n_samples, pad, bos, eos, temperature, top_k, seed).generate(src)` returns
(B, n_samples, max_len) int64:

  * sample s of source b starts from BOS and appends one drawn token per step; a row ends at its first drawn EOS or PAD
    (kept) or when it holds max_len tokens; PAD behind.  Rows end individually.
  * the token drawn at column t is argmax_v z_v over the candidate set, z_v = logit_v / T + g_v, equal z to the lower id
    (Gumbel-max: distributed as softmax(logits / T) restricted to the candidates).  Candidates: the whole vocabulary for
    top_k = 0, else the top_k largest logits, ties at the boundary to the lower id.
  * g_v = -log(-log(u)), u = ((x >> 9) * 2 + 1) * 2^-24, x = word v & 3 of Philox4x32-10 at counter (t, s, v >> 2, 0) and
    key (lo32(key_b), hi32(key_b)); key_b = FNV-1a-64 over the 8 little-endian bytes of the seed, then the 4 little-endian
    bytes of every non-PAD token of src[b] in column order.

The decoder is rerun on the whole prefix every step (no cache), which is what a causal decoder's last position gives.
`generate` also records, per row and column, the gaps the GPU tests judge a divergence by: best-to-second z among the
candidates and the top_k-th to (top_k + 1)-th logit.
"""
from __future__ import annotations

import math

import numpy as np
import torch

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK32 = 0xFFFFFFFF


def philox4x32_10(ctr, key) -> np.ndarray:
    """Vectorised Philox4x32-10: ctr (4, ...) and key (2, ...) of 32-bit values (broadcast) -> (4, ...) uint64 holding
    32-bit words."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK32 for x in ctr]
    k0, k1 = (np.asarray(x, dtype=np.uint64) & _MASK32 for x in key)
    c = list(np.broadcast_arrays(*c, k0, k1))
    k0, k1 = c[4].copy(), c[5].copy()
    c = [x.copy() for x in c[:4]]
    for _ in range(10):
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & np.uint64(_MASK32)
        hi1, lo1 = p1 >> np.uint64(32), p1 & np.uint64(_MASK32)
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(_W0)) & np.uint64(_MASK32)
        k1 = (k1 + np.uint64(_W1)) & np.uint64(_MASK32)
    return np.stack(c)


def source_key(src_row, seed: int, pad: int) -> int:
    """FNV-1a-64 over the seed's 8 little-endian bytes and the 4 little-endian bytes of every non-PAD token."""
    h = 0xcbf29ce484222325
    data = int(seed).to_bytes(8, "little") + b"".join(
        (int(t) & _MASK32).to_bytes(4, "little") for t in src_row if int(t) != pad)
    for byte in data:
        h = ((h ^ byte) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h


def gumbel_noise(t: int, s, key, V: int) -> torch.Tensor:
    """(R, V) float32 Gumbel noise of column t for rows with sample indices s (R,) and keys (R,)."""
    s = np.asarray(s, dtype=np.uint64)[:, None]
    key = np.asarray(key, dtype=np.uint64)[:, None]
    v = np.arange(V, dtype=np.uint64)[None, :]
    words = philox4x32_10((np.uint64(t), s, v >> np.uint64(2), np.uint64(0)),
                          (key & np.uint64(_MASK32), key >> np.uint64(32)))          # (4, R, V)
    x = np.take_along_axis(words, (v & np.uint64(3)).astype(np.int64)[None].repeat(words.shape[1], 1), axis=0)[0]
    u = torch.from_numpy(((x >> np.uint64(9)) * np.uint64(2) + np.uint64(1)).astype(np.float32)) * (2.0 ** -24)
    return -torch.log(-torch.log(u))


def candidate_mask(logits: torch.Tensor, top_k: int) -> torch.Tensor:
    """(R, V) bool: the top_k largest logits of every row, ties at the boundary to the lower token id."""
    R, V = logits.shape
    if top_k == 0 or top_k >= V:
        return torch.ones(R, V, dtype=torch.bool)
    order = torch.from_numpy(np.lexsort((np.arange(V)[None].repeat(R, 0), -logits.numpy()), axis=-1))   # value desc, id asc
    mask = torch.zeros(R, V, dtype=torch.bool)
    mask.scatter_(1, order[:, :top_k], True)
    return mask


def draw(logits: torch.Tensor, t: int, s, keys, temperature: float, top_k: int):
    """One step for rows (R, V) of fp32 logits -> (tokens (R,), z gap (R,), k gap (R,))."""
    R, V = logits.shape
    cand = candidate_mask(logits, top_k)
    z = logits / torch.full_like(logits, temperature) + gumbel_noise(t, s, keys, V)
    z = torch.where(cand, z, torch.full_like(z, -math.inf))
    best = z.max(dim=1).values
    ids = torch.arange(V).expand(R, V)
    tok = torch.where(z == best[:, None], ids, torch.full_like(ids, V)).min(dim=1).values
    zs = z.sort(dim=1, descending=True).values
    zgap = (zs[:, 0] - zs[:, 1]) if V > 1 else torch.full((R,), math.inf)
    zgap = torch.where(torch.isfinite(zgap), zgap, torch.full_like(zgap, math.inf))
    if 0 < top_k < V:
        ls = logits.sort(dim=1, descending=True).values
        kgap = ls[:, top_k - 1] - ls[:, top_k]
    else:
        kgap = torch.full((R,), math.inf)
    return tok, zgap, kgap


class TranslationInferenceSampling:
    def __init__(self, model, max_len: int, n_samples: int, pad_token: int, bos_token: int, eos_token: int,
                 temperature: float = 1.0, top_k: int = 0, seed: int = 0):
        self.model, self.max_len, self.n_samples = model, max_len, n_samples
        self.pad_token, self.bos_token, self.eos_token = pad_token, bos_token, eos_token
        self.temperature, self.top_k, self.seed = temperature, top_k, seed
        self.model_calls_num = 0
        self.given_tokens = 0
        self.sampled_tokens = 0
        self.unfinished = 0
        self.zgap = None      # (B, S, max_len) gaps of the draw that filled each column (inf where nothing was drawn)
        self.kgap = None

    def generate(self, src: torch.Tensor, seed: int | None = None) -> torch.Tensor:
        seed = self.seed if seed is None else seed
        m, S, L = self.model, self.n_samples, self.max_len
        B = src.shape[0]
        R = B * S
        src_pad = m.src_pad_token_i
        keys = np.array([source_key(src[b].tolist(), seed, src_pad) for b in range(B)], dtype=np.uint64).repeat(S)
        s_idx = np.tile(np.arange(S, dtype=np.uint64), B)
        pad_mask = src == src_pad
        self.given_tokens += int((~pad_mask).sum())
        memory = m.encode_src(src, pad_mask).repeat_interleave(S, 0)
        mem_mask = pad_mask.repeat_interleave(S, 0)
        tokens = torch.full((R, L), self.pad_token, dtype=torch.int64)
        tokens[:, 0] = self.bos_token
        zgap = torch.full((R, L), math.inf)
        kgap = torch.full((R, L), math.inf)
        live = torch.ones(R, dtype=torch.bool)
        for t in range(1, L):
            idx = live.nonzero()[:, 0]
            if idx.numel() == 0:
                break
            logits = m.decode_tgt(tokens[idx, :t], memory[idx], mem_mask[idx])[:, -1, :].float()
            self.model_calls_num += 1
            tok, zg, kg = draw(logits, t, s_idx[idx.numpy()], keys[idx.numpy()], self.temperature, self.top_k)
            tokens[idx, t] = tok
            zgap[idx, t], kgap[idx, t] = zg, kg
            self.sampled_tokens += int(idx.numel())
            ended = (tok == self.eos_token) | (tok == self.pad_token)
            if t == L - 1:
                self.unfinished += int((~ended).sum())
            live[idx[ended]] = False
        self.zgap, self.kgap = zgap.view(B, S, L), kgap.view(B, S, L)
        return tokens.view(B, S, L)
