"""Sampling decoding on the B200 (TranslationInferenceSampling / ttb_sample_generate) against the CPU oracle
(oracle/sampling.py).

Draws follow the oracle's noise bit for bit, but the logits they act on carry the precision of their path (DESIGN.md
section 5), and log() on the device and on the CPU may differ in the last bit.  So a row may diverge from the oracle only
at a column where the oracle's best-to-second z gap is below 2 x (logit tolerance) / T + 1e-5, or where its top_k-th to
(top_k + 1)-th logit gap is below 2 x (logit tolerance); the rest of such a row is not compared.  Logit tolerance: 2e-5 on
the fp32 path, max(1.5e-2, 1e-2 max|logit|) on the bf16 path against the oracle's bf16 emulation."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from helpers import ARCH
from oracle.sampling import TranslationInferenceSampling as SamplingOracle
from oracle.transformer import OracleTransformer
from translation_transformer_b200 import TranslationScorer, _lib
from translation_transformer_b200.decoding import TranslationInferenceGreedy, TranslationInferenceSampling
from translation_transformer_b200.weights import ModelConfig, random_init_state_dict

pytestmark = pytest.mark.gpu

PAD, BOS, EOS = 0, 1, 2
FP32_LOGIT = 2e-5
REPO = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _weights(arch, V, seed=11, eos_bias=0.9):
    cfg = ModelConfig(src_vocab_size=V, tgt_vocab_size=V, **ARCH[arch])
    sd = {k: v.clone() for k, v in random_init_state_dict(cfg, seed).items()}
    sd["next_token_classifier.bias"][EOS] += eos_bias
    sd["next_token_classifier.bias"][PAD] -= 5.0
    return cfg, sd


def _engine(cfg, sd, precision):
    from translation_transformer_b200.model import B200Transformer
    return B200Transformer(cfg, sd, precision=precision, device=0)


def _src(B, Ls, V, seed):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(3, V, (B, Ls), generator=g)
    src[:, 0] = BOS
    for b in range(B):
        n = int(torch.randint(2, Ls + 1, (1,), generator=g))
        src[b, n:] = PAD
    return src


def _sampler(eng, max_len, S, T, k, seed):
    return TranslationInferenceSampling(eng, max_len, S, PAD, BOS, EOS, temperature=T, top_k=k, seed=seed)


def _check_against_oracle(out, ref, oracle, T, logit_tol):
    """Every row equals the oracle's up to its first differing column, which must be a near-tie; returns the number of
    diverged rows."""
    z_tol, k_tol = 2 * logit_tol / T + 1e-5, 2 * logit_tol
    B, S, L = ref.shape
    diverged = 0
    for b in range(B):
        for s in range(S):
            diff = (out[b, s] != ref[b, s]).nonzero()
            if diff.numel() == 0:
                continue
            c = int(diff[0])
            zg, kg = float(oracle.zgap[b, s, c]), float(oracle.kgap[b, s, c])
            assert zg < z_tol or kg < k_tol, (b, s, c, zg, kg, out[b, s].tolist(), ref[b, s].tolist())
            diverged += 1
    return diverged


def _row_lengths(out):
    """Drawn tokens of every row: up to and including the first EOS or PAD, else max_len - 1."""
    body = out[..., 1:]
    L1 = body.shape[-1]
    idx = torch.arange(1, L1 + 1).expand_as(body)
    first = torch.where((body == EOS) | (body == PAD), idx, torch.full_like(idx, L1 + 1)).amin(-1)
    return first.clamp(max=L1)


@pytest.mark.parametrize("top_k", [0, 5, 20])
@pytest.mark.parametrize("T", [1.0, 0.7])
@pytest.mark.parametrize("arch", ["small", "full"])
def test_fp32_matches_oracle(dev, arch, T, top_k):
    V, L, S = 53, 24, 4
    cfg, sd = _weights(arch, V)
    src = _src(3, 17, V, seed=top_k + 1)
    oracle = SamplingOracle(OracleTransformer(sd, cfg.num_heads), L, S, PAD, BOS, EOS, T, top_k, seed=77)
    ref = oracle.generate(src)
    eng = _engine(cfg, sd, "fp32")
    try:
        gen = _sampler(eng, L, S, T, top_k, 77)
        out = gen.generate(src.to(dev)).cpu()
    finally:
        eng.close()
    assert out.shape == (3, S, L) and out.dtype == torch.int64
    n = _row_lengths(ref)
    assert len(set(n.view(-1).tolist())) > 1, "rows should end at different steps"
    if _check_against_oracle(out, ref, oracle, T, FP32_LOGIT) == 0:
        assert gen.model_calls_num == oracle.model_calls_num
        assert gen.sampled_tokens == oracle.sampled_tokens
        assert gen.last_stats.unfinished == oracle.unfinished
    assert gen.given_tokens == oracle.given_tokens


@pytest.mark.parametrize("top_k", [0, 5, 20])
@pytest.mark.parametrize("no_fused", [False, True], ids=["fused", "forced_fallback"])
def test_bf16_matches_oracle_emulation(dev, no_fused, top_k, monkeypatch):
    """The fused draw (top_k 0 and 5; top_k = 20 takes the fallback by itself) and the logits GEMM + sample_rows_kernel."""
    if no_fused:
        monkeypatch.setenv("TTB_NO_FUSED_ARGMAX", "1")
    V, L, S, T = 288, 20, 3, 1.0
    cfg, sd = _weights("full", V)
    src = _src(3, 21, V, seed=5)
    om = OracleTransformer(sd, cfg.num_heads, gemm_dtype="bf16")
    scale = float(om(src, torch.full((3, 1), BOS)).abs().max())
    tol = max(1.5e-2, 1e-2 * scale)
    oracle = SamplingOracle(om, L, S, PAD, BOS, EOS, T, top_k, seed=3)
    ref = oracle.generate(src)
    eng = _engine(cfg, sd, "bf16")
    try:
        out = _sampler(eng, L, S, T, top_k, 3).generate(src.to(dev)).cpu()
    finally:
        eng.close()
    _check_against_oracle(out, ref, oracle, T, tol)
    # the first draw of every row sees logits within tol of the oracle's: nearly all rows agree there
    agree = (out[..., 1] == ref[..., 1]).float().mean()
    assert agree >= 0.5, agree


def _chi2_p(counts, probs):
    from scipy.stats import chisquare
    exp = probs * counts.sum()
    order = np.argsort(-exp)
    obs_b, exp_b, acc_o, acc_e = [], [], 0.0, 0.0
    for i in order:                     # pool the bins with small expectations into one
        if exp[i] >= 5:
            obs_b.append(counts[i]); exp_b.append(exp[i])
        else:
            acc_o += counts[i]; acc_e += exp[i]
    if acc_e > 0:
        obs_b.append(acc_o); exp_b.append(acc_e)
    obs_b, exp_b = np.array(obs_b, dtype=np.float64), np.array(exp_b, dtype=np.float64)
    exp_b *= obs_b.sum() / exp_b.sum()
    return float(chisquare(obs_b, exp_b).pvalue)


@pytest.mark.parametrize("top_k", [0, 5])
def test_first_token_distribution(dev, top_k):
    V, T = 53, 0.7
    cfg, sd = _weights("small", V, eos_bias=0.0)
    src = _src(1, 15, V, seed=8)
    om = OracleTransformer(sd, cfg.num_heads)
    logits = om(src, torch.full((1, 1), BOS))[0, -1].double()
    eng = _engine(cfg, sd, "fp32")
    try:
        first = []
        for seed in (1, 2, 3, 4):
            out = _sampler(eng, 2, 2048, T, top_k, seed).generate(src.to(dev)).cpu()
            first.append(out[0, :, 1])
    finally:
        eng.close()
    first = torch.cat(first)
    counts = np.bincount(first.numpy(), minlength=V).astype(np.float64)
    z = logits / T
    if top_k:
        top = torch.topk(logits, top_k).indices
        outside = torch.ones(V, dtype=torch.bool)
        outside[top] = False
        assert counts[outside.numpy()].sum() == 0
        z = torch.where(outside, torch.full_like(z, -float("inf")), z)
    probs = torch.softmax(z, 0).numpy()
    p = _chi2_p(counts, probs)
    assert p > 1e-4, p


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_top_k_1_equals_greedy(dev, precision):
    V, L, S = 288, 40, 3
    cfg, sd = _weights("full", V)
    src = _src(8, 25, V, seed=13)
    eng = _engine(cfg, sd, precision)
    try:
        greedy = TranslationInferenceGreedy(eng, L, PAD, BOS, EOS).generate(src.to(dev)).cpu()[:, 0]
        out = _sampler(eng, L, S, 0.5, 1, 99).generate(src.to(dev)).cpu()
    finally:
        eng.close()
    for b in range(src.shape[0]):
        g = greedy[b]
        end = next((i for i in range(1, L) if int(g[i]) in (EOS, PAD)), L - 1)
        for s in range(S):
            assert torch.equal(out[b, s, :end + 1], g[:end + 1]), (b, s)
            assert bool((out[b, s, end + 1:] == PAD).all())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_invariance(dev, precision):
    V, L, S = 288, 30, 4
    cfg, sd = _weights("full", V)
    src = _src(6, 23, V, seed=17)
    src[4] = src[1]                      # duplicate source
    eng = _engine(cfg, sd, precision)
    try:
        gen = _sampler(eng, L, S, 1.0, 0, 5)
        full = gen.generate(src.to(dev)).cpu()
        again = gen.generate(src.to(dev)).cpu()
        singles = [gen.generate(src[b:b + 1].to(dev)).cpu() for b in range(6)]
        perm = torch.tensor([3, 0, 5, 1, 4, 2])
        permuted = gen.generate(src[perm].to(dev)).cpu()
        other_seed = gen.generate(src.to(dev), seed=6).cpu()
    finally:
        eng.close()
    assert torch.equal(full, again)
    for b in range(6):
        assert torch.equal(full[b], singles[b][0]), b
    assert torch.equal(permuted, full[perm])
    assert torch.equal(full[4], full[1])
    assert not torch.equal(other_seed, full)
    assert len({tuple(r) for r in full.view(-1, L).tolist()}) > 1


def test_graph_cache_does_not_go_stale(dev):
    """One engine alternating temperatures, top_k, seeds and greedy decoding; every call equals a fresh engine's."""
    V, L, S = 288, 24, 3
    cfg, sd = _weights("full", V)
    src = _src(4, 19, V, seed=23)
    calls = [("s", 1.0, 0, 1), ("s", 0.6, 0, 1), ("g",), ("s", 1.0, 5, 1), ("s", 1.0, 0, 2), ("s", 0.6, 5, 2), ("g",), ("s", 1.0, 0, 1)]

    def run(eng, c):
        if c[0] == "g":
            return TranslationInferenceGreedy(eng, L, PAD, BOS, EOS).generate(src.to(dev)).cpu()
        return _sampler(eng, L, S, c[1], c[2], c[3]).generate(src.to(dev)).cpu()

    eng = _engine(cfg, sd, "bf16")
    try:
        shared = [run(eng, c) for c in calls]
    finally:
        eng.close()
    for c, got in zip(calls, shared):
        fresh = _engine(cfg, sd, "bf16")
        try:
            assert torch.equal(got, run(fresh, c)), c
        finally:
            fresh.close()
    assert not torch.equal(shared[0], shared[1]) and not torch.equal(shared[0], shared[4])
    assert torch.equal(shared[0], shared[7])


def test_c_abi_rejects_bad_arguments_and_scorer_takes_the_output(dev):
    V, L, S = 53, 16, 3
    cfg, sd = _weights("small", V, eos_bias=2.0)
    src = _src(2, 11, V, seed=2).to(dev)
    eng = _engine(cfg, sd, "fp32")
    try:
        out = torch.zeros(2 * 1100 * L, dtype=torch.int64, device=dev)
        st = _lib.GenerateStats()
        bad = [dict(n=0), dict(n=1025), dict(T=0.0), dict(T=float("inf")), dict(T=float("nan")), dict(k=-1), dict(k=V + 1),
               dict(L=1), dict(eos=PAD), dict(L=1023)]
        for b in bad:
            a = dict(n=S, T=1.0, k=0, L=L, eos=EOS, **{})
            a.update(b)
            rc = eng.lib.ttb_sample_generate(eng._h, src.data_ptr(), 2, 11, a["L"], a["n"], a["T"], a["k"], 7, PAD, BOS, a["eos"],
                                             out.data_ptr(), C.byref(st), C.c_void_p(0))
            assert rc == 2, (b, rc)
        samples = _sampler(eng, L, S, 1.0, 0, 7).generate(src)
        r = TranslationScorer(eng, PAD, EOS).score(src, samples)
    finally:
        eng.close()
    assert torch.equal(r.n_tokens.cpu().long(), _row_lengths(samples.cpu()))
    assert bool((r.logp <= 0).all())


def test_predict_csv_is_identical_across_in_flight_engines(tmp_path):
    outs = []
    for k in (1, 3):
        out = tmp_path / f"pred_{k}.csv"
        cmd = [sys.executable, str(REPO / "scripts" / "predict.py"), "--synthetic", "96", "--batch-size", "16", "--generation", "sampling",
               "--n-samples", "3", "--temperature", "0.8", "--top-k", "5", "--sampling-seed", "11", "--max-len", "40",
               "--in-flight", str(k), "--output", str(out)]
        r = subprocess.run(cmd, cwd=str(REPO), capture_output=True, text=True, timeout=900, env={**os.environ, "PYTHONPATH": str(REPO)})
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        outs.append(out.read_bytes())
    assert outs[0] == outs[1]
    assert b"prediction_3" in outs[0].splitlines()[0]
