"""Teacher-forced scoring on the B200 (TranslationScorer / ttb_score_targets) against the CPU oracle (oracle/scoring.py).

Tolerances follow from the logit contract of DESIGN.md section 5: a log-probability moves by at most its own logit's error
plus the largest logit error, so 2 x 2e-5 per token on the fp32 path and 2 x max(1.5e-2, 1e-2 max|logit|) on the bf16 path
(against the oracle's bf16 emulation)."""
from __future__ import annotations

import ctypes as C

import pytest
import torch

from helpers import ARCH
from oracle.scoring import score as oracle_score
from oracle.transformer import OracleTransformer
from translation_transformer_b200 import TranslationScorer
from translation_transformer_b200.weights import ModelConfig, random_init_state_dict

pytestmark = pytest.mark.gpu

PAD, BOS, EOS = 0, 1, 2
FP32_TOK = 4e-5


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _weights(arch, V, seed=11):
    cfg = ModelConfig(src_vocab_size=V, tgt_vocab_size=V, **ARCH[arch])
    sd = {k: v.clone() for k, v in random_init_state_dict(cfg, seed).items()}
    sd["next_token_classifier.bias"][EOS] += 0.9
    sd["next_token_classifier.bias"][PAD] -= 5.0
    return cfg, sd


def _engine(cfg, sd, precision):
    from translation_transformer_b200.model import B200Transformer
    return B200Transformer(cfg, sd, precision=precision, device=0)


def _inputs(B, K, Ls, Lt, V, seed):
    """Ragged sources and candidates: EOS in the middle with random tokens or PAD behind it, PAD tails without EOS,
    candidates that run to Lt, and candidates with PAD in column 1."""
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(3, V, (B, Ls), generator=g)
    src[:, 0] = BOS
    for b in range(B):
        n = int(torch.randint(2, Ls + 1, (1,), generator=g))
        src[b, n:] = PAD
    tgt = torch.randint(3, V, (B, K, Lt), generator=g)
    tgt[:, :, 0] = BOS
    for b in range(B):
        for k in range(K):
            kind = (b * K + k) % 5
            e = int(torch.randint(1, Lt, (1,), generator=g))
            if kind == 0:
                tgt[b, k, e] = EOS                      # random tokens behind the EOS
            elif kind == 1:
                tgt[b, k, e] = EOS
                tgt[b, k, e + 1:] = PAD
            elif kind == 2:
                tgt[b, k, e:] = PAD                     # PAD tail, no EOS
            elif kind == 4 and b % 2 == 0:
                tgt[b, k, 1:] = PAD                     # nothing to score
    return src, tgt


def _randomise_tails(tgt, n, V, seed):
    g = torch.Generator().manual_seed(seed)
    out = tgt.clone()
    Lt = tgt.shape[-1]
    for idx in torch.cartesian_prod(*[torch.arange(s) for s in tgt.shape[:-1]]).view(-1, tgt.dim() - 1):
        lo = min(int(n[tuple(idx)]) + 2, Lt)    # the column behind the end stays (a terminating PAD must stay PAD)
        out[tuple(idx)][lo:] = torch.randint(0, V, (Lt - lo,), generator=g)
    return out


def _score(eng, src, tgt, dev, per_token=True):
    r = TranslationScorer(eng, PAD, EOS).score(src.to(dev), tgt.to(dev), per_token=per_token)
    return tuple(x.cpu() if x is not None else None for x in r)


@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("arch", ["small", "full"])
def test_fp32_matches_oracle(dev, arch, K):
    V = 53
    cfg, sd = _weights(arch, V)
    src, tgt = _inputs(5, K, 37, 23, V, seed=K)
    ref = oracle_score(OracleTransformer(sd, cfg.num_heads), src, tgt, PAD, EOS)
    eng = _engine(cfg, sd, "fp32")
    try:
        logp, n, tok = _score(eng, src, tgt, dev)
    finally:
        eng.close()
    assert torch.equal(n, ref[1])
    assert (tok - ref[2]).abs().max() <= FP32_TOK
    assert ((logp - ref[0]).abs() <= FP32_TOK * n.clamp(min=1)).all()
    assert bool((tok[n == 0] == 0).all()) and bool((logp[n == 0] == 0).all())


@pytest.mark.parametrize("arch,V,no_fused", [("full", 288, False), ("full", 288, True), ("full", 600, False), ("small", 288, False)],
                         ids=["fused", "forced_fallback", "vocab_above_512", "small"])
def test_bf16_matches_oracle_emulation(dev, arch, V, no_fused, monkeypatch):
    """The fused vocabulary projection + statistics kernel (full architecture, V = 288), and the logits GEMM +
    logprob_stats fallback: forced, for a vocabulary the fused kernel does not take, and at E = 64, where the kernel's
    exchange area does not fit its operand tiles."""
    if no_fused:
        monkeypatch.setenv("TTB_NO_FUSED_STATS", "1")
    cfg, sd = _weights(arch, V)
    src, tgt = _inputs(4, 3, 41, 29, V, seed=7)
    om = OracleTransformer(sd, cfg.num_heads, gemm_dtype="bf16")
    ref = oracle_score(om, src, tgt, PAD, EOS)
    scale = float(om(src.repeat_interleave(3, 0), tgt.view(-1, 29)).abs().max())
    tol = 2 * max(1.5e-2, 1e-2 * scale)
    eng = _engine(cfg, sd, "bf16")
    try:
        logp, n, tok = _score(eng, src, tgt, dev)
    finally:
        eng.close()
    assert torch.equal(n, ref[1])
    assert (tok - ref[2]).abs().max() <= tol, ((tok - ref[2]).abs().max(), tol)
    assert ((logp - ref[0]).abs() <= tol * n.clamp(min=1)).all()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_tokens_behind_the_end_change_nothing(dev, precision):
    V = 288
    cfg, sd = _weights("full", V)
    src, tgt = _inputs(6, 4, 45, 31, V, seed=3)
    eng = _engine(cfg, sd, precision)
    try:
        a = _score(eng, src, tgt, dev)
        changed = _randomise_tails(tgt, a[1], V, seed=4)
        assert not torch.equal(changed, tgt)
        b = _score(eng, src, changed, dev)
    finally:
        eng.close()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_shared_encoder_equals_repeated_sources(dev):
    V = 53
    cfg, sd = _weights("full", V)
    B, K, Lt = 4, 5, 27
    src, tgt = _inputs(B, K, 33, Lt, V, seed=9)
    eng = _engine(cfg, sd, "fp32")
    try:
        a = _score(eng, src, tgt, dev)
        b = _score(eng, src.repeat_interleave(K, 0), tgt.reshape(B * K, 1, Lt), dev)
    finally:
        eng.close()
    assert torch.equal(a[1], b[1].view(B, K))
    assert (a[2] - b[2].view(B, K, Lt - 1)).abs().max() <= 1e-6
    assert (a[0] - b[0].view(B, K)).abs().max() <= 1e-6 * max(1, int(a[1].max()))


def test_greedy_outputs_score_as_teacher_forced_argmax(dev):
    from translation_transformer_b200.decoding import TranslationInferenceGreedy
    V = 53
    cfg, sd = _weights("small", V)
    src, _ = _inputs(6, 1, 30, 2, V, seed=12)
    eng = _engine(cfg, sd, "fp32")
    try:
        out = TranslationInferenceGreedy(eng, 40, PAD, BOS, EOS).generate(src.to(dev)).cpu()   # (B, 1, 40)
        logp, n, tok = _score(eng, src, out, dev)
    finally:
        eng.close()
    assert bool((out[:, :, 0] == BOS).all()) and int(n.sum()) > 0
    om = OracleTransformer(sd, cfg.num_heads)
    best = torch.log_softmax(om(src, out[:, 0]), dim=-1).amax(dim=-1)[:, :-1]       # max log-softmax at every position
    for b in range(src.shape[0]):
        m = int(n[b, 0])
        assert (tok[b, 0, :m] >= best[b, :m] - FP32_TOK).all(), b


def test_chunked_call_equals_per_source_calls(dev):
    """64 sources x 10 candidates x 60 columns = 38400 decoder rows: two chunks of whole sources."""
    V = 53
    cfg, sd = _weights("small", V)
    src, tgt = _inputs(64, 10, 21, 60, V, seed=21)
    eng = _engine(cfg, sd, "fp32")
    try:
        a = _score(eng, src, tgt, dev)
        per = [_score(eng, src[b:b + 1], tgt[b:b + 1], dev) for b in range(64)]
        with pytest.raises(ValueError, match="32768"):
            TranslationScorer(eng, PAD, EOS).score(src[:1].to(dev), torch.full((1, 40, 1000), 5, device=dev))
        # the C ABI refuses it as well, before any device work
        out = torch.zeros(40, device=dev)
        rc = eng.lib.ttb_score_targets(eng._h, src[:1].to(dev).data_ptr(), 1, 21, out.data_ptr(), 40, 1000, PAD, EOS, out.data_ptr(),
                                       out.data_ptr(), None, C.c_void_p(0))
        assert rc != 0 and "32768" in eng.lib.ttb_last_error().decode()
    finally:
        eng.close()
    assert torch.equal(a[1], torch.cat([p[1] for p in per]))
    assert (a[2] - torch.cat([p[2] for p in per])).abs().max() <= FP32_TOK
    assert (a[0] - torch.cat([p[0] for p in per])).abs().max() <= FP32_TOK * int(a[1].max())


def test_bf16_repeated_calls_are_bitwise_equal(dev):
    V = 288
    cfg, sd = _weights("full", V)
    src, tgt = _inputs(32, 5, 60, 48, V, seed=5)
    eng = _engine(cfg, sd, "bf16")
    try:
        a = _score(eng, src, tgt, dev)
        b = _score(eng, src, tgt, dev)
    finally:
        eng.close()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_two_dimensional_targets_and_cpu_inputs(dev):
    V = 53
    cfg, sd = _weights("small", V)
    src, tgt = _inputs(3, 1, 19, 17, V, seed=2)
    eng = _engine(cfg, sd, "fp32")
    try:
        r3 = TranslationScorer(eng, PAD, EOS).score(src.to(dev), tgt.to(dev))
        r2 = TranslationScorer(eng, PAD, EOS).score(src, tgt[:, 0], per_token=True)
    finally:
        eng.close()
    assert r3.token_logp is None and r3.logp.shape == (3, 1) and r3.logp.is_cuda
    assert r2.logp.shape == (3,) and r2.n_tokens.dtype == torch.int32 and r2.token_logp.shape == (3, 16) and not r2.logp.is_cuda
    assert torch.equal(r2.logp, r3.logp[:, 0].cpu()) and torch.equal(r2.n_tokens, r3.n_tokens[:, 0].cpu())
