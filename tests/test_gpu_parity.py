"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Everything goes through the C ABI of
libttb200 via the package's reference-shaped Python interface and is compared with
  * the golden vectors produced by the unmodified reference (tests/golden/), and
  * the CPU oracle (oracle/) on fresh seeded inputs.
Bit-exact for tokens / accepted lengths / draft indices; logits within the tolerance written
in each test (1e-5 class for the fp32 path, 1e-2 for bf16)."""
import numpy as np
import pytest
import torch

from helpers import case_weights, load_json, load_npz, test_file_sources
from translation_transformer_b200.weights import ModelConfig, random_init_state_dict

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _engine(cfg, sd, precision):
    from translation_transformer_b200.model import B200Transformer
    return B200Transformer(cfg, sd, precision=precision, device=0)


# ---------------------------------------------------------------------------------------------
def test_make_drafts_matches_reference_golden(dev):
    from translation_transformer_b200.utils.drafting import make_drafts
    cases, dz, meta = load_json("drafts.json"), load_npz("drafts.npz"), load_json("model_forward.json")
    _, src, _ = test_file_sources(meta["vocab"])
    src = src.to(dev)
    syn = torch.from_numpy(dz["syn_src"].astype(np.int64)).to(dev)
    for c in cases:
        if c.get("synthetic"):
            s = syn[:, 1:]
        else:
            s = src[:c["B"]] if c["with_bos"] else src[:c["B"], 1:]
        d = make_drafts(s, c["D"], c["N"], c["min_draft_len"], c["max_draft_len"], c["eos"], c["pad"], c["replace"])
        assert d.dtype == torch.int64 and d.is_cuda
        assert np.array_equal(d.cpu().numpy(), dz[f"d{c['id']}"].astype(np.int64)), c


def test_make_drafts_reference_test_grid_vs_oracle(dev):
    """All 1008 size combinations of the reference's own test (tests/test_drafting.py:19-61) on its source file: requested
    shape (what the reference asserts) and bit-exact agreement with the oracle."""
    from oracle.drafting import make_drafts as oracle_drafts
    from test_oracle_golden import REF_GRID_AMOUNTS, REF_GRID_BATCHES, REF_GRID_LENGTHS
    from translation_transformer_b200.utils.drafting import make_drafts
    meta = load_json("model_forward.json")
    tk, src, _ = test_file_sources(meta["vocab"])
    src_d = src.to(dev)
    eos, pad, rep = tk.eos_token_idx, tk.pad_token_idx, tk.encoder_dict["c"]
    for B in REF_GRID_BATCHES:
        for n_drafts in REF_GRID_LENGTHS:
            for draft_len in REF_GRID_AMOUNTS:
                got = make_drafts(src_d[:B], draft_len, n_drafts, 1, 200, eos, pad, rep)
                assert tuple(got.shape) == (min(B, src.shape[0]), n_drafts, draft_len)
                ref = oracle_drafts(src[:B].numpy(), draft_len, n_drafts, 1, 200, eos, pad, rep)
                assert np.array_equal(got.cpu().numpy(), ref), (B, n_drafts, draft_len)


def test_make_drafts_argument_checks(dev):
    from translation_transformer_b200.utils.drafting import make_drafts
    s = torch.tensor([[5, 6, 7, 2, 0]], device=dev)
    for args in ((2, 0, 1, 10, 2, 0, 5), (2, 1, 5, 4, 2, 0, 5), (2, 1, 1, 10, 2, 0, 0), (2, 1, 1, 10, 2, 0, 2), (2, 1, 1, 10, 2, 2, 5)):
        with pytest.raises(AssertionError):
            make_drafts(s, *args)


def test_make_drafts_random_vs_oracle(dev):
    from oracle.drafting import make_drafts as oracle_drafts
    from translation_transformer_b200.utils.drafting import make_drafts
    g = torch.Generator().manual_seed(7)
    for trial in range(40):
        B = int(torch.randint(1, 9, (1,), generator=g))
        L = int(torch.randint(2, 220, (1,), generator=g))
        src = torch.zeros(B, L, dtype=torch.int64)
        for b in range(B):
            n = int(torch.randint(0, L, (1,), generator=g))
            src[b, :n] = torch.randint(3, 300, (n,), generator=g)
            src[b, n] = 2
        D = int(torch.randint(1, 60, (1,), generator=g))
        N = int(torch.randint(1, 70, (1,), generator=g))
        ref = oracle_drafts(src.numpy(), D, N, 1, 200, 2, 0, 9)
        got = make_drafts(src.to(dev), D, N, 1, 200, 2, 0, 9).cpu().numpy()
        assert np.array_equal(ref, got), (B, L, D, N)


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["small", "full"])
def test_forward_fp32_matches_reference_golden(dev, name):
    z, meta = load_npz("model_forward.npz"), load_json("model_forward.json")
    m = meta["meta"][name]
    cfg = ModelConfig(**m["config"])
    eng = _engine(cfg, random_init_state_dict(cfg, m["seed"]), "fp32")
    src, tgt = torch.from_numpy(z[name + "_src"]).to(dev), torch.from_numpy(z[name + "_tgt"]).to(dev)
    pad = src == 0
    mem = eng.encode_src(src, pad).cpu()
    ref_mem = torch.from_numpy(z[name + "_memory"])
    assert (mem - ref_mem)[~pad.cpu()].abs().max() < 2e-5          # fp32 tolerance
    logits = eng.decode_tgt(tgt, ref_mem.to(dev), pad).cpu()
    assert (logits - torch.from_numpy(z[name + "_logits"])).abs().max() < 2e-5
    full = eng(src, tgt).cpu()
    assert (full - torch.from_numpy(z[name + "_forward_logits"])).abs().max() < 2e-5
    eng.close()


def test_gemm_fp32_vs_torch(dev):
    import ctypes as C
    from translation_transformer_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(3)
    for (M, N, K, relu) in ((1, 30, 64, 0), (77, 300, 256, 1), (253, 768, 256, 0), (130, 256, 2048, 0)):
        A = torch.randn(M, K, generator=g).to(dev)
        W = torch.randn(N, K, generator=g).to(dev)
        b = torch.randn(N, generator=g).to(dev)
        Cm = torch.empty(M, N, device=dev)
        _lib.check(lib.ttb_gemm(0, A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, relu, None), "ttb_gemm")
        ref = A.double() @ W.double().t() + b.double()
        if relu:
            ref = ref.clamp_min(0)
        assert (Cm.double() - ref).abs().max() < 1e-3 * (K ** 0.5) / 16


# ---------------------------------------------------------------------------------------------
def _greedy_cases():
    return load_json("greedy_speculative.json")


@pytest.mark.parametrize("case", _greedy_cases(), ids=lambda c: c["id"])
def test_greedy_speculative_fp32_matches_reference_golden(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    z = load_npz("greedy_speculative.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceGreedySpeculative(eng, case["max_len"], case["draft_len"], case["n_drafts"], 0, 1, 2,
                                                case["replace"], keep_trace=True)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    err = None
    try:
        out = gen.generate(src)
    except RuntimeError as e:
        err = "RuntimeError"
        msg = str(e)
    assert err == case["error"], (err, case["error"])
    if err is None:
        assert out.shape == (case["B"], 1, case["max_len"]) and out.dtype == torch.int64
        assert np.array_equal(out.cpu().numpy(), z[case["id"] + "_out"].astype(np.int64))   # bit-exact tokens
        assert gen.model_calls_num == case["model_calls"]
    else:
        # the reference fails inside iteration `model_calls` (after the decoder call for the
        # shape error, before it for the index error); the engine stops at the same iteration
        assert gen.model_calls_num in (case["model_calls"], case["model_calls"] - 1), (gen.model_calls_num, case["model_calls"], msg)
    ref_nacc = z[case["id"] + "_nacc"].reshape(-1, case["n_drafts"])
    ref_pick = z[case["id"] + "_pick"]
    nacc = np.array([a for t in gen.trace for a in t["n_accepted"]], dtype=np.int64)
    pick = np.array([p for t in gen.trace for p in t["draft_index"]], dtype=np.int64)
    n = len(pick)
    assert n <= len(ref_pick) and (err is not None or n == len(ref_pick))
    assert np.array_equal(pick, ref_pick[:n])                                   # bit-exact draft indices
    assert np.array_equal(nacc, ref_nacc[np.arange(n), ref_pick[:n]])           # bit-exact accepted lengths
    assert [len(t["rows"]) for t in gen.trace] == case["rows_per_iter"][:len(gen.trace)]
    eng.close()


def test_greedy_speculative_fp32_vs_oracle_fresh_inputs(dev):
    """Seeded inputs that are not in the fixtures: synthetic ragged sources, vocab 300."""
    from oracle.greedy_speculative import GreedySpeculativeOracle
    from oracle.transformer import OracleTransformer
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    from helpers import SMALL
    cfg = ModelConfig(src_vocab_size=300, tgt_vocab_size=300, **SMALL)
    for seed, eos_bias, B, max_len, D, N in ((101, 0.9, 6, 90, 8, 9), (102, 1.0, 9, 70, 4, 25), (103, 0.8, 3, 120, 12, 2)):
        sd = {k: v.clone() for k, v in random_init_state_dict(cfg, seed).items()}
        sd["tgt_token_featurizer.embedding.weight"] = sd["src_token_featurizer.embedding.weight"]
        sd["next_token_classifier.bias"][2] += eos_bias
        sd["next_token_classifier.bias"][0] -= 5.0
        g = torch.Generator().manual_seed(seed)
        lens = torch.randint(10, 80, (B,), generator=g)
        src = torch.zeros(B, int(lens.max()) + 2, dtype=torch.int64)
        for b in range(B):
            n = int(lens[b])
            src[b, 0] = 1
            src[b, 1:n + 1] = torch.randint(4, 300, (n,), generator=g)
            src[b, n + 1] = 2
        oracle = GreedySpeculativeOracle(OracleTransformer(sd, cfg.num_heads), max_len, D, N, 0, 1, 2, 7, keep_trace=True)
        eng = _engine(cfg, sd, "fp32")
        gen = TranslationInferenceGreedySpeculative(eng, max_len, D, N, 0, 1, 2, 7, keep_trace=True)
        try:
            ref = oracle.generate(src)
        except RuntimeError:
            with pytest.raises(RuntimeError):
                gen.generate(src.to(dev))
            continue
        out = gen.generate(src.to(dev))
        assert np.array_equal(out.cpu().numpy(), ref.numpy())
        assert gen.model_calls_num == oracle.model_calls_num
        assert [t["n_accepted"] for t in gen.trace] == [t["n_accepted"] for t in oracle.trace]
        assert [t["draft_index"] for t in gen.trace] == [t["draft_index"] for t in oracle.trace]
        eng.close()


# ---------------------------------------------------------------------------------------------
# bf16 path: tcgen05 GEMMs.  Tolerances: GEMM vs fp32 matmul of the same bf16 operands 2e-3
# (accumulation order only); logits vs the fp32 reference atol=rtol=1e-2 (north_star bf16 bound).
def test_gemm_bf16_tcgen05_vs_torch(dev):
    from translation_transformer_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(4)
    shapes = ((128, 128, 64, 0), (1, 30, 64, 0), (77, 288, 256, 1), (253, 768, 256, 0), (130, 256, 2048, 0),
              (8096, 2048, 256, 1), (1000, 512, 256, 0), (300, 300, 128, 0), (129, 129, 192, 1))
    for (M, N, K, relu) in shapes:
        A = torch.randn(M, K, generator=g).to(dev).bfloat16()
        W = (torch.randn(N, K, generator=g) * 0.1).to(dev).bfloat16()
        b = torch.randn(N, generator=g).to(dev)
        Cm = torch.full((M, N), float("nan"), device=dev)
        _lib.check(lib.ttb_gemm(1, A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, relu, None), "ttb_gemm")
        torch.cuda.synchronize()
        ref = A.float().double() @ W.float().double().t() + b.double()
        if relu:
            ref = ref.clamp_min(0)
        err = (Cm.double() - ref).abs().max().item()
        assert err < 2e-3, (M, N, K, relu, err)
    # bf16 result: K = 256 and N a multiple of 384 / 256 run on the CTA-pair kernel (cta_group::2) from 1024 rows on,
    # the other shapes on the persistent kernel; error bound = bf16 rounding of the result
    for (M, N, K, relu) in ((8096, 768, 256, 0), (2000, 768, 256, 1), (1025, 512, 256, 0), (1300, 1536, 256, 0), (700, 768, 256, 0), (3000, 256, 256, 0)):
        A = torch.randn(M, K, generator=g).to(dev).bfloat16()
        W = (torch.randn(N, K, generator=g) * 0.1).to(dev).bfloat16()
        b = torch.randn(N, generator=g).to(dev)
        Cm = torch.full((M, N), float("nan"), device=dev, dtype=torch.bfloat16)
        _lib.check(lib.ttb_gemm_bf16_out(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, relu, None), "ttb_gemm_bf16_out")
        torch.cuda.synchronize()
        ref = A.float().double() @ W.float().double().t() + b.double()
        if relu:
            ref = ref.clamp_min(0)
        err = ((Cm.double() - ref).abs() / (1.0 + ref.abs())).max().item()
        assert err < 6e-3, (M, N, K, relu, err)


@pytest.mark.parametrize("name", ["small", "full"])
def test_forward_bf16_within_tolerance(dev, name):
    from oracle.transformer import OracleTransformer
    z, meta = load_npz("model_forward.npz"), load_json("model_forward.json")
    m = meta["meta"][name]
    cfg = ModelConfig(**m["config"])
    sd = random_init_state_dict(cfg, m["seed"])
    eng = _engine(cfg, sd, "bf16")
    src, tgt = torch.from_numpy(z[name + "_src"]).to(dev), torch.from_numpy(z[name + "_tgt"]).to(dev)
    full = eng(src, tgt).cpu()
    ref = torch.from_numpy(z[name + "_forward_logits"])
    # bf16 tolerance: 1e-2 of the logit scale.  Rounding the weights alone to bf16 already moves the
    # logits of this random-init model by up to 8e-3 (rms 3e-3), see DESIGN.md "precision contract".
    assert (full - ref).abs().max() <= 1e-2 * ref.abs().max(), ((full - ref).abs().max(), ref.abs().max())
    assert torch.allclose(full, ref, atol=1.5e-2, rtol=1e-2), (full - ref).abs().max()
    # against the oracle run under the same precision contract only accumulation-order noise remains,
    # amplified where it flips a bf16 rounding
    emu = OracleTransformer(sd, cfg.num_heads, gemm_dtype="bf16")(src.cpu(), tgt.cpu())
    assert torch.allclose(full, emu, atol=1.5e-2, rtol=1e-2), (full - emu).abs().max()
    eng.close()


def _check_tokens_near_argmax(oracle_model, src, out, pad, eos, margin):
    """Every emitted token must be an argmax of the fp32 reference logits up to `margin`
    (teacher-forced on the emitted prefix); returns the number of positions checked."""
    checked = 0
    for b in range(out.shape[0]):
        row = out[b, 0]
        if (row == eos).sum() == 0:
            continue                       # unfinished queries come back as all-PAD rows
        n = int((row == eos).nonzero()[0]) + 1
        s = src[b:b + 1]
        mem = oracle_model.encode_src(s, s == 0)
        logits = oracle_model.decode_tgt(row[:n].unsqueeze(0), mem, s == 0)[0]
        for i in range(n - 1):
            chosen = logits[i, row[i + 1]]
            assert chosen >= logits[i].max() - margin, (b, i, float(chosen), float(logits[i].max()))
            checked += 1
    return checked


def test_greedy_speculative_bf16_tokens_are_reference_argmax(dev):
    from oracle.transformer import OracleTransformer
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    z = load_npz("greedy_speculative.npz")
    total = 0
    for case in load_json("greedy_speculative.json"):
        if case["error"] is not None or "eos_bias" not in case:
            continue
        cfg, sd = case_weights(case)
        eng = _engine(cfg, sd, "bf16")
        gen = TranslationInferenceGreedySpeculative(eng, case["max_len"], case["draft_len"], case["n_drafts"], 0, 1, 2,
                                                    case["replace"], keep_trace=True)
        src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64))
        try:
            out = gen.generate(src.to(dev)).cpu()
        except RuntimeError:
            eng.close()
            continue                       # a near-tie flipped a token into one of the reference's own failure modes
        total += _check_tokens_near_argmax(OracleTransformer(sd, cfg.num_heads), src, out, 0, 2, margin=3e-2)
        # internal consistency of the speculative bookkeeping
        produced = {}
        for t in gen.trace:
            for q, a in zip(t["rows"], t["n_accepted"]):
                produced[q] = produced.get(q, 0) + a + 1
        for b in range(out.shape[0]):
            row = out[b, 0]
            if (row == 2).any():
                assert produced[b] == int((row == 2).nonzero()[0])
        eng.close()
    assert total > 200


def _ragged_sources(B, lo, hi, vocab, seed):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(lo, hi, (B,), generator=g)
    src = torch.zeros(B, int(lens.max()) + 2, dtype=torch.int64)
    for b in range(B):
        n = int(lens[b])
        src[b, 0] = 1
        src[b, 1:n + 1] = torch.randint(4, vocab, (n,), generator=g)
        src[b, n + 1] = 2
    return src


@pytest.mark.parametrize("D,N,lo,hi", [(10, 23, 10, 60), (20, 7, 20, 50), (6, 30, 200, 236)],
                         ids=["bench-shape", "long-drafts", "long-sources"])
def test_greedy_speculative_bf16_full_size_fused_kernels(dev, D, N, lo, hi, monkeypatch):
    """The benchmark model shape (E=256, F=2048: fused GEMM+LayerNorm, fused FFN, fused classifier+argmax, tensor-core
    attention with KV cache) through the whole decoding loop, against the fp32 path of the same engine code (which is
    bit-exact with the reference, see the fp32 tests).  A random-init model of this size never emits EOS at a useful
    length, so the comparison is on the per-iteration trace (accepted length and chosen draft of every query): bf16
    may only leave the fp32 trajectory through a near-tie of two logits, i.e. late or never.  TTB_NO_FUSED_ARGMAX=1 is
    read per call: set after a graph-replayed call on the same engine, it recaptures the graph with the logits GEMM and
    arg-max kernel, whose trace follows the fused one under the same near-tie rule."""
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    from helpers import FULL
    vocab, B, max_len = 120, 5, 72
    cfg = ModelConfig(src_vocab_size=vocab, tgt_vocab_size=vocab, **FULL)
    sd = {k: v.clone() for k, v in random_init_state_dict(cfg, 4242).items()}
    sd["tgt_token_featurizer.embedding.weight"] = sd["src_token_featurizer.embedding.weight"]
    src = _ragged_sources(B, lo, hi, vocab, seed=77 + D)
    traces, calls, outs = {}, {}, {}
    for prec in ("fp32", "bf16"):
        eng = _engine(cfg, sd, prec)
        gen = TranslationInferenceGreedySpeculative(eng, max_len, D, N, 0, 1, 2, 7, keep_trace=True)
        try:
            outs[prec] = gen.generate(src.to(dev)).cpu()
        except RuntimeError:
            outs[prec] = None
        traces[prec] = [(t["rows"], t["n_accepted"], t["draft_index"]) for t in gen.trace]
        calls[prec] = gen.model_calls_num
        if prec == "bf16" and outs[prec] is not None:
            # the graph-replayed loop (no trace) must give the same tokens as the traced, eagerly launched one
            gen2 = TranslationInferenceGreedySpeculative(eng, max_len, D, N, 0, 1, 2, 7)
            out2 = gen2.generate(src.to(dev)).cpu()
            assert np.array_equal(outs[prec].numpy(), out2.numpy())
            assert gen2.model_calls_num == calls[prec]
            monkeypatch.setenv("TTB_NO_FUSED_ARGMAX", "1")
            for keep_trace in (False, True):
                gen3 = TranslationInferenceGreedySpeculative(eng, max_len, D, N, 0, 1, 2, 7, keep_trace=keep_trace)
                try:
                    gen3.generate(src.to(dev))
                except RuntimeError:
                    pass                   # a near-tie flipped a token into one of the reference's own failure modes
                if keep_trace:
                    traces["bf16_unfused"] = [(t["rows"], t["n_accepted"], t["draft_index"]) for t in gen3.trace]
                else:              # two launches (logits GEMM, arg-max) where the fused kernel made one
                    assert gen3.gpu_launches / gen3.model_calls_num > gen2.gpu_launches / gen2.model_calls_num
            monkeypatch.delenv("TTB_NO_FUSED_ARGMAX")
        eng.close()
    def near_tie_only(a, b):
        n = min(len(traces[a]), len(traces[b]))
        first_diff = next((i for i in range(n) if traces[a][i] != traces[b][i]), None)
        assert n >= 5
        assert first_diff is None or first_diff >= 8, (a, b, first_diff, traces[a][first_diff], traces[b][first_diff])
        return n, first_diff

    n, first_diff = near_tie_only("fp32", "bf16")
    if "bf16_unfused" in traces:
        near_tie_only("bf16", "bf16_unfused")
    if first_diff is None:
        assert calls["fp32"] == calls["bf16"]
        if outs["fp32"] is not None and outs["bf16"] is not None:
            assert np.array_equal(outs["fp32"].numpy(), outs["bf16"].numpy())
    print(f"bf16 trace identical to fp32 for {n if first_diff is None else first_diff} of {n} iterations")


# ---------------------------------------------------------------------------------------------
# speculative beam search (configs[2], configs[3] of BASELINE.json at test size)
def _beam_cases():
    return load_json("beam_speculative.json")


@pytest.mark.parametrize("case", _beam_cases(), ids=lambda c: c["id"])
def test_beam_speculative_fp32_matches_reference_golden(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("beam_speculative.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                    case["vocab"], False, 0, 1, 2, case["C_token"], keep_trace=True)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    out = gen.generate(src).cpu().numpy()
    ref = z[case["id"] + "_out"].astype(np.int64)
    assert out.shape == ref.shape
    assert np.array_equal(out, ref)                                                    # all hypotheses, best first, bit-exact
    assert (gen.model_calls_num, gen.accepted_tokens_num, gen.produced_non_pad_tokens) == \
        (case["model_calls"], case["accepted_tokens"], case["produced_non_pad_tokens"])
    nacc = np.concatenate([t["n_accepted"].reshape(-1) for t in gen.trace])
    pick = np.concatenate([t["pick"] for t in gen.trace])
    assert np.array_equal(nacc, z[case["id"] + "_nacc"].astype(np.int64))               # accepted lengths of every draft
    assert np.array_equal(pick, z[case["id"] + "_pick"].astype(np.int64))               # chosen draft indices
    # no trace: steady-state iterations are enqueued ahead of the host reading the outcome of the one before
    # (engine.cu:beam_api): same hypotheses and counters, also on the second call on the same engine
    for _ in range(2):
        gen2 = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                         case["vocab"], False, 0, 1, 2, case["C_token"])
        assert np.array_equal(gen2.generate(src).cpu().numpy(), ref)
        assert (gen2.model_calls_num, gen2.accepted_tokens_num, gen2.produced_non_pad_tokens) == \
            (case["model_calls"], case["accepted_tokens"], case["produced_non_pad_tokens"])
    eng.close()


def _beam_smart_cases():
    return load_json("beam_smart.json")


@pytest.mark.parametrize("case", _beam_smart_cases(), ids=lambda c: c["id"])
def test_beam_speculative_smart_drafts_fp32_matches_reference_golden(dev, case):
    """smart_drafts_mode=True (speculative_decoding.py:600-845): hypotheses, counters, accepted length of every tried
    draft (ragged groups padded with -1 like the reference's topk_in_each_group) and the chosen drafts, bit-exact."""
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("beam_smart.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                    case["vocab"], True, 0, 1, 2, case["C_token"], keep_trace=True)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    if case["error"] is not None:
        with pytest.raises(AssertionError):
            gen.generate(src)
        eng.close()
        return
    out = gen.generate(src).cpu().numpy()
    ref = z[case["id"] + "_out"].astype(np.int64)
    assert out.shape == ref.shape
    assert np.array_equal(out, ref)
    assert (gen.model_calls_num, gen.accepted_tokens_num, gen.produced_non_pad_tokens) == \
        (case["model_calls"], case["accepted_tokens"], case["produced_non_pad_tokens"])
    ref_nacc, ref_pick = z[case["id"] + "_nacc"].astype(np.int64), z[case["id"] + "_pick"].astype(np.int64)
    o_n = o_p = 0
    assert len(gen.trace) == len(case["topk1_shapes"])
    for t, (C, L) in zip(gen.trace, case["topk1_shapes"]):
        na = t["n_accepted"]
        assert na.shape[0] == C
        assert np.array_equal(na[:, :L], ref_nacc[o_n:o_n + C * L].reshape(C, L))
        assert (na[:, L:] == -1).all()
        assert np.array_equal(t["pick"], ref_pick[o_p:o_p + C])
        o_n += C * L
        o_p += C
    for _ in range(2):   # no trace: iterations enqueued ahead, also on the second call on the same engine
        gen2 = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                         case["vocab"], True, 0, 1, 2, case["C_token"])
        assert np.array_equal(gen2.generate(src).cpu().numpy(), ref)
        assert (gen2.model_calls_num, gen2.accepted_tokens_num, gen2.produced_non_pad_tokens) == \
            (case["model_calls"], case["accepted_tokens"], case["produced_non_pad_tokens"])
    eng.close()


def test_beam_speculative_smart_drafts_bf16_runs(dev):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("beam_smart.npz")
    case = [c for c in _beam_smart_cases() if c["id"] == "smart1"][0]
    cfg, sd = case_weights(case)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    eng = _engine(cfg, sd, "bf16")
    gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                    case["vocab"], True, 0, 1, 2, case["C_token"])
    out = gen.generate(src).cpu().numpy()
    ref = z[case["id"] + "_out"].astype(np.int64)
    assert out.shape[:2] == ref.shape[:2]
    same = sum(int(out.shape[2] == ref.shape[2] and np.array_equal(out[b, 0], ref[b, 0])) for b in range(ref.shape[0]))
    assert same >= ref.shape[0] // 2, (same, ref.shape[0])
    eng.close()


def test_beam_speculative_bf16_runs_and_is_consistent(dev):
    """bf16 hypotheses may differ from fp32 at near-ties; check structure and that the best hypothesis
    of most queries matches the fp32 engine."""
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("beam_speculative.npz")
    case = [c for c in _beam_cases() if c["id"] == "beam1"][0]
    cfg, sd = case_weights(case)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    outs = {}
    for prec in ("fp32", "bf16"):
        eng = _engine(cfg, sd, prec)
        gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                        case["vocab"], False, 0, 1, 2, case["C_token"])
        outs[prec] = gen.generate(src).cpu()
        eng.close()
    a, b = outs["fp32"], outs["bf16"]
    assert a.shape[:2] == b.shape[:2] == (case["B"], case["n_best"])
    assert (b[:, :, 0] == 1).all()
    w = min(a.shape[2], b.shape[2])
    same_top1 = sum(bool(torch.equal(a[i, 0, :w], b[i, 0, :w])) for i in range(case["B"]))
    assert same_top1 >= case["B"] // 2


# ---------------------------------------------------------------------------------------------
# standard (non-speculative) decoding, standard_decoding.py
def _standard_cases(kind):
    return [c for c in load_json("standard_decoding.json") if c["kind"] == kind]


@pytest.mark.parametrize("case", _standard_cases("greedy"), ids=lambda c: c["id"])
def test_standard_greedy_fp32_matches_reference_golden(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceGreedy
    z = load_npz("standard_decoding.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceGreedy(eng, case["max_len"], 0, 1, 2)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64))
    out = gen.generate(src.to(dev)).cpu()
    assert np.array_equal(out.numpy(), z[case["id"] + "_out"].astype(np.int64))
    assert gen.model_calls_num == case["model_calls"] and gen.given_tokens == case["given_tokens"]
    # second call on the same engine (graph replay, buffers reused)
    out2 = gen.generate(src.to(dev)).cpu()
    assert np.array_equal(out.numpy(), out2.numpy())
    eng.close()


def test_standard_greedy_bf16_tokens_are_reference_argmax(dev):
    from oracle.transformer import OracleTransformer
    from translation_transformer_b200.decoding import TranslationInferenceGreedy
    z = load_npz("standard_decoding.npz")
    total = 0
    for case in _standard_cases("greedy"):
        if "eos_bias" not in case:
            continue
        cfg, sd = case_weights(case)
        eng = _engine(cfg, sd, "bf16")
        src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64))
        out = TranslationInferenceGreedy(eng, case["max_len"], 0, 1, 2).generate(src.to(dev)).cpu()
        total += _check_tokens_near_argmax(OracleTransformer(sd, cfg.num_heads), src, out, 0, 2, margin=3e-2)
        eng.close()
    assert total > 100


@pytest.mark.parametrize("case", _standard_cases("beam"), ids=lambda c: c["id"])
def test_standard_beam_search_fp32_matches_reference_golden(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    z = load_npz("standard_decoding.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceBeamSearch(eng, case["beam_size"], case["max_len"], 0, 1, 2)
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64))
    out = gen.generate(src.to(dev)).cpu()
    ref = z[case["id"] + "_out"].astype(np.int64)
    assert tuple(out.shape) == tuple(ref.shape)
    assert np.array_equal(out.numpy(), ref)
    assert gen.model_calls_num == case["model_calls"] and gen.given_tokens == case["given_tokens"]
    eng.close()


def test_standard_beam_search_bf16_runs_and_is_consistent(dev):
    """bf16 hypotheses may differ from fp32 at near-ties; the best hypothesis of most queries must agree."""
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    z = load_npz("standard_decoding.npz")
    same = total = 0
    for case in _standard_cases("beam"):
        cfg, sd = case_weights(case)
        src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64))
        eng = _engine(cfg, sd, "bf16")
        out = TranslationInferenceBeamSearch(eng, case["beam_size"], case["max_len"], 0, 1, 2).generate(src.to(dev)).cpu().numpy()
        eng.close()
        ref = z[case["id"] + "_out"].astype(np.int64)
        assert out.shape[:2] == ref.shape[:2]
        for b in range(ref.shape[0]):
            w = min(out.shape[2], ref.shape[2])
            same += int(np.array_equal(out[b, 0, :w], ref[b, 0, :w]) and out.shape[2] == ref.shape[2])
            total += 1
    assert same >= 0.7 * total, (same, total)


def test_ffn_pair_kernel_matches_cta_group1_kernel(dev):
    """The CTA-pair feed-forward kernel (cta_group::2, clusters of four, chained out-projection, A operand in tensor
    memory) and the cta_group::1 kernel + separate out-projection kernel give bit-identical logits: golden inputs, a
    ragged batch, and a batch with more 256-row blocks than co-resident clusters (each mode in its own process)."""
    import subprocess
    import sys
    from pathlib import Path
    script = Path(__file__).resolve().parent.parent / "scripts" / "ffn_pair_check.py"
    r = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "WORST 0.0" in r.stdout


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("generation", ["greedy_speculative", "beam_search_speculative"])
def test_batches_in_flight_give_the_sequential_predictions(dev, generation):
    """pipeline.py / `predict_batches`: three batches decoded concurrently by three engines (own streams, workspaces and
    CUDA graphs) return, in order, exactly what `predict_step` returns batch by batch (bf16 benchmark model shape)."""
    from helpers import FULL
    from translation_transformer_b200.lightning_model import VanillaEncoderDecoderTransformerLightning
    import importlib.util
    from pathlib import Path
    spec = importlib.util.spec_from_file_location("predict_driver", Path(__file__).resolve().parent.parent / "scripts" / "predict.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    vocab = 96
    tk = mod.synthetic_tokenizer(vocab)
    model = VanillaEncoderDecoderTransformerLightning(
        src_tokenizer=tk, tgt_tokenizer=tk, generation=generation, beam_size=3, max_len=40, n_drafts=5, draft_len=6,
        smart_drafts_mode=False, report_prediction_time=False, precision="bf16", device=0, seed=99, batches_in_flight=3, **FULL)
    batches = [{"src_tokens": _ragged_sources(4 if i % 2 else 3, 12, 30, vocab, seed=500 + i)} for i in range(7)]

    def run(fn):
        try:
            return fn()
        except RuntimeError as ex:      # the reference's own failure modes are results too
            return str(ex)[:40]

    seq = [run(lambda b=b, i=i: model.predict_step({"src_tokens": b["src_tokens"].to(dev)}, i).cpu()) for i, b in enumerate(batches)]
    calls_seq = model._counter("model_calls_num")
    par = [p if isinstance(p, str) else p.cpu() for p in model.predict_batches(batches, on_error=lambda i, ex: str(ex)[:40])]
    assert model._counter("model_calls_num") == 2 * calls_seq
    assert sum(g.model_calls_num > 0 for g in model.generators) >= 2      # the batches really went to several engines
    assert len(par) == len(seq)
    for a, b in zip(seq, par):
        assert type(a) is type(b)
        assert a == b if isinstance(a, str) else torch.equal(a, b)
    for m in model.models:
        m.close()


def test_lightning_checkpoint_state_dict_loads(dev):
    """A reference Lightning checkpoint's `state_dict` (keys prefixed `model.`, plus the non-persistent positional buffer that
    some exports carry) goes through `load_checkpoint_state_dict` (lightning_model.py:73 of the reference builds the same
    prefix) and decodes like an engine built from the plain state dict."""
    from translation_transformer_b200.data_handling import ChemSMILESTokenizer
    from translation_transformer_b200.lightning_model import VanillaEncoderDecoderTransformerLightning
    from translation_transformer_b200.model import sinusoid_table
    from helpers import SMALL
    meta = load_json("model_forward.json")
    tk, src, _ = test_file_sources(meta["vocab"])
    cfg = ModelConfig(src_vocab_size=tk.n_tokens, tgt_vocab_size=tk.n_tokens, **SMALL)
    sd = {k: v.clone() for k, v in random_init_state_dict(cfg, 33).items()}
    sd["next_token_classifier.bias"][2] += 0.5
    sd["next_token_classifier.bias"][0] -= 5.0
    kw = dict(src_tokenizer=tk, tgt_tokenizer=tk, generation="greedy_speculative", max_len=60, n_drafts=5, draft_len=6, precision="fp32",
              share_embeddings=False, **SMALL)
    a = VanillaEncoderDecoderTransformerLightning(state_dict=sd, **kw)
    b = VanillaEncoderDecoderTransformerLightning(seed=5, **kw)                 # other weights first
    ckpt = {"model." + k: v for k, v in sd.items()}
    ckpt["model.positional_encoding.pe"] = sinusoid_table(SMALL["embedding_dim"], 5000)
    b.load_checkpoint_state_dict(ckpt)
    batch = {"src_tokens": src[:4].to(dev)}
    ra, rb = a.predict_step(batch, 0), b.predict_step(batch, 0)
    assert torch.equal(ra, rb) and (ra != 0).any()
    for m in a.models + b.models:
        m.close()
