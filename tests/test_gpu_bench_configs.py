"""GPU parity AT THE BENCHMARKED CONFIGURATIONS (BASELINE.json configs[1..3]): the exact workloads bench.py times,
against goldens produced by the unmodified reference (tests/golden/make_golden_bench.py -> bench_configs.{npz,json}).

  fp32 engine : bit-exact tokens / hypotheses, accepted lengths of every draft, chosen draft indices, call counts
  bf16 engine : (the path the benchmark runs) the fraction of queries whose token sequence equals the reference's is
                measured, printed (and recorded as a junit property) and asserted against the bound written in each test
"""
import json

import numpy as np
import pytest
import torch

from helpers import GOLDEN, load_json, load_npz
from translation_transformer_b200.synthetic import synthetic_sources
from translation_transformer_b200.weights import (ModelConfig, PRODUCT_PREDICTION, SINGLE_STEP_RETRO, copy_task_state_dict,
                                                  random_init_state_dict, state_dict_checksum)

pytestmark = pytest.mark.gpu
ARCH = {"product": PRODUCT_PREDICTION, "retro": SINGLE_STEP_RETRO}


def _cases(kind):
    if not (GOLDEN / "bench_configs.json").exists():
        return []
    return [c for c in load_json("bench_configs.json") if c["kind"] == kind]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _weights(case):
    cfg = ModelConfig(src_vocab_size=case["vocab"], tgt_vocab_size=case["vocab"], **ARCH[case["arch"]])
    sd = copy_task_state_dict(cfg, case["seed"]) if case["weights"] == "copy" else random_init_state_dict(cfg, case["seed"])
    assert state_dict_checksum(sd) == case["checksum"], "weights differ from the ones the golden run used (torch CPU RNG / arithmetic drifted)"
    return cfg, sd


def _sources(case, z):
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64))
    if "file_line" in case:      # BASELINE.json configs[0]: one line of the reference's test file (tokenized by make_golden_bench.py)
        return src
    # the fixture's sources ARE the bench's batches: regenerate them the way bench.py does and compare
    n = 32 if case["arch"] == "product" else case["B"]
    again = synthetic_sources(n, case["vocab"], seed=case["src_seed"], **case.get("src_kw", {}))[:case["B"]]
    assert torch.equal(src, again)
    return src


def _engine(cfg, sd, precision):
    from translation_transformer_b200.model import B200Transformer
    return B200Transformer(cfg, sd, precision=precision, device=0)


@pytest.mark.parametrize("case", _cases("greedy"), ids=lambda c: c["id"])
def test_greedy_bench_config_fp32_bit_exact(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    z = load_npz("bench_configs.npz")
    cfg, sd = _weights(case)
    src = _sources(case, z).to(dev)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceGreedySpeculative(eng, case["max_len"], case["draft_len"], case["n_drafts"], 0, 1, 2, 7, keep_trace=True)
    assert case["error"] is None
    out = gen.generate(src).cpu().numpy()
    ref = z[case["id"] + "_out"].astype(np.int64)
    assert np.array_equal(out, ref)                                                   # bit-exact tokens, all 32 queries
    assert gen.model_calls_num == case["model_calls"]
    ref_nacc = z[case["id"] + "_nacc"].astype(np.int64).reshape(-1, case["n_drafts"])
    ref_pick = z[case["id"] + "_pick"].astype(np.int64)
    nacc = np.array([a for t in gen.trace for a in t["n_accepted"]], dtype=np.int64)
    pick = np.array([p for t in gen.trace for p in t["draft_index"]], dtype=np.int64)
    assert len(pick) == len(ref_pick)
    assert np.array_equal(pick, ref_pick)                                             # chosen draft of every (iteration, query)
    assert np.array_equal(nacc, ref_nacc[np.arange(len(pick)), ref_pick])             # its accepted length
    assert [len(t["rows"]) for t in gen.trace] == case["rows_per_iter"]               # retirement: live queries per iteration
    if case["weights"] == "copy":
        assert (ref != 0).any(-1).all(), "every query of the trained-like workload finishes with a non-empty prediction"
    eng.close()


@pytest.mark.parametrize("case", _cases("greedy"), ids=lambda c: c["id"])
def test_greedy_bench_config_bf16_vs_reference(dev, case, record_property):
    """The benchmarked path itself (bf16, CUDA graphs, fused kernels) against the reference's tokens."""
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    z = load_npz("bench_configs.npz")
    cfg, sd = _weights(case)
    src = _sources(case, z).to(dev)
    eng = _engine(cfg, sd, "bf16")
    ref = z[case["id"] + "_out"].astype(np.int64)
    ref_nacc = z[case["id"] + "_nacc"].astype(np.int64).reshape(-1, case["n_drafts"])
    ref_pick = z[case["id"] + "_pick"].astype(np.int64)
    ref_acc = ref_nacc[np.arange(len(ref_pick)), ref_pick]
    # (a) traced run (no CUDA graph): accepted length per (iteration, query) against the reference
    gen = TranslationInferenceGreedySpeculative(eng, case["max_len"], case["draft_len"], case["n_drafts"], 0, 1, 2, 7, keep_trace=True)
    out_t = gen.generate(src).cpu().numpy()
    nacc = np.array([a for t in gen.trace for a in t["n_accepted"]], dtype=np.int64)
    n = min(len(nacc), len(ref_acc))
    first_diff = int(np.argmax(nacc[:n] != ref_acc[:n])) if (nacc[:n] != ref_acc[:n]).any() else n
    cells_equal = float((nacc[:n] == ref_acc[:n]).mean())
    # (b) the graph-replayed run the benchmark times
    gen2 = TranslationInferenceGreedySpeculative(eng, case["max_len"], case["draft_len"], case["n_drafts"], 0, 1, 2, 7)
    out = gen2.generate(src).cpu().numpy()
    assert np.array_equal(out, out_t), "graph-replayed and eagerly launched loops disagree"
    same = (out[:, 0] == ref[:, 0]).all(-1)
    frac = float(same.mean())
    report = {"case": case["id"], "queries_identical_to_reference": frac, "n_queries": int(len(same)),
              "accepted_length_cells_equal": cells_equal, "first_differing_cell": first_diff, "cells": int(n),
              "decoder_calls": gen2.model_calls_num, "reference_decoder_calls": case["model_calls"]}
    print("bf16 vs reference:", json.dumps(report))
    record_property("bf16_vs_reference", json.dumps(report))
    if case["weights"] == "copy":
        # trained-like margins: bf16 reproduces the reference tokens except at genuine near-ties
        assert frac >= 0.9, report
        assert gen2.model_calls_num == case["model_calls"] or frac < 1.0
    else:
        # random-init logits have many near-ties (top-2 margins of 1e-3 are common), so the bf16 trajectory leaves the
        # fp32 one after some iterations; the bookkeeping up to there must be identical and the run must terminate
        # the way the reference does (all-PAD rows for unfinished queries)
        assert first_diff >= 32, report
        assert np.array_equal(out == 0, ref == 0) or frac < 1.0
    eng.close()


@pytest.mark.parametrize("case", _cases("beam"), ids=lambda c: c["id"])
def test_beam_bench_config_fp32_bit_exact(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("bench_configs.npz")
    cfg, sd = _weights(case)
    src = _sources(case, z).to(dev)
    eng = _engine(cfg, sd, "fp32")
    gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"], case["vocab"],
                                                    bool(case.get("smart", False)), 0, 1, 2, 7, keep_trace=True)
    assert case["error"] is None
    out = gen.generate(src).cpu().numpy()
    ref = z[case["id"] + "_out"].astype(np.int64)
    assert out.shape == ref.shape
    assert np.array_equal(out, ref)                                                   # all n_best hypotheses of every query
    assert (gen.model_calls_num, gen.accepted_tokens_num, gen.produced_non_pad_tokens) == \
        (case["model_calls"], case["accepted_tokens"], case["produced_non_pad_tokens"])
    pick = np.concatenate([t["pick"] for t in gen.trace])
    assert np.array_equal(pick, z[case["id"] + "_pick"].astype(np.int64))
    ref_nacc = z[case["id"] + "_nacc"].astype(np.int64)
    if case.get("smart"):    # ragged draft groups: the reference pads each iteration to its widest group, the engine to n_drafts
        off = 0
        assert len(gen.trace) == len(case["topk1_shapes"])
        for t, (C, L) in zip(gen.trace, case["topk1_shapes"]):
            na = t["n_accepted"]
            assert na.shape[0] == C and np.array_equal(na[:, :L], ref_nacc[off:off + C * L].reshape(C, L)) and (na[:, L:] == -1).all()
            off += C * L
    else:
        assert np.array_equal(np.concatenate([t["n_accepted"].reshape(-1) for t in gen.trace]), ref_nacc)
    eng.close()


@pytest.mark.parametrize("case", _cases("beam"), ids=lambda c: c["id"])
def test_beam_bench_config_bf16_vs_reference(dev, case, record_property):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("bench_configs.npz")
    cfg, sd = _weights(case)
    src = _sources(case, z).to(dev)
    eng = _engine(cfg, sd, "bf16")
    gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"], case["vocab"],
                                                    bool(case.get("smart", False)), 0, 1, 2, 7)
    out = gen.generate(src).cpu().numpy()
    ref = z[case["id"] + "_out"].astype(np.int64)
    W = max(out.shape[-1], ref.shape[-1])
    o = np.zeros(out.shape[:2] + (W,), np.int64); o[..., :out.shape[-1]] = out
    r = np.zeros(ref.shape[:2] + (W,), np.int64); r[..., :ref.shape[-1]] = ref
    top1 = float((o[:, 0] == r[:, 0]).all(-1).mean())
    # hypothesis SETS per query (bf16 may swap the order of two hypotheses whose scores differ by < 1e-2)
    set_frac = float(np.mean([len({tuple(h) for h in o[b]} & {tuple(h) for h in r[b]}) / ref.shape[1] for b in range(ref.shape[0])]))
    report = {"case": case["id"], "top1_identical": top1, "hypotheses_in_common": set_frac, "decoder_calls": gen.model_calls_num,
              "reference_decoder_calls": case["model_calls"], "accepted_tokens": gen.accepted_tokens_num,
              "reference_accepted_tokens": case["accepted_tokens"]}
    print("bf16 vs reference:", json.dumps(report))
    record_property("bf16_vs_reference", json.dumps(report))
    assert top1 >= 0.75 and set_frac >= 0.6, report
    eng.close()


@pytest.mark.parametrize("case", [c for c in _cases("beam") if c["n_best"] <= 16], ids=lambda c: c["id"])
def test_fused_classifier_statistics_match_the_unfused_kernels(dev, case, monkeypatch):
    """csrc/gemm_tcgen05.cu:classifier_stats_kernel (vocabulary projection + soft-max statistics + n_best largest logits
    straight from tensor memory) against the logits GEMM + beam.cu:beam_stats_kernel it replaces on the bf16 path: the same
    hypotheses, decoder calls and acceptance counters (the two differ only in the order of the soft-max sum)."""
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz("bench_configs.npz")
    cfg, sd = _weights(case)
    src = _sources(case, z).to(dev)
    res = {}
    monkeypatch.setenv("TTB_FUSED_STATS_WIDE", "1")      # n_best > 8 runs unfused by default (slower fused); exercised here
    for flag in ("1", "0"):
        monkeypatch.setenv("TTB_NO_FUSED_STATS", flag)
        eng = _engine(cfg, sd, "bf16")
        gen = TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"], case["vocab"],
                                                        bool(case.get("smart", False)), 0, 1, 2, 7, keep_trace=True)
        out = gen.generate(src).cpu().numpy()
        res[flag] = (out, gen.model_calls_num, gen.accepted_tokens_num, gen.gpu_launches,
                     np.concatenate([t["n_accepted"].reshape(-1) for t in gen.trace]))
        eng.close()
    (o_un, c_un, a_un, l_un, n_un), (o_fu, c_fu, a_fu, l_fu, n_fu) = res["1"], res["0"]
    assert l_fu < l_un                                   # one launch less per iteration
    same = o_un.shape == o_fu.shape and np.array_equal(o_un, o_fu)
    print(f"{case['id']}: fused vs unfused statistics: identical={same}, calls {c_fu}/{c_un}, accepted {a_fu}/{a_un}, launches {l_fu}/{l_un}")
    assert c_fu == c_un and np.array_equal(n_fu, n_un)   # accepted length of every draft in every iteration
    assert o_un.shape == o_fu.shape and (o_un[:, 0] == o_fu[:, 0]).all()          # best hypothesis of every query
    assert (o_un == o_fu).all(-1).mean() >= 0.95         # the rest up to swaps of hypotheses whose scores differ in the last bits


@pytest.mark.parametrize("n_best,smart", [(1, False), (3, False), (8, False), (5, True)])
def test_fused_classifier_statistics_other_beam_widths(dev, n_best, smart, monkeypatch):
    """Fused against unfused statistics for list lengths around the register list of the fused kernel (8 entries) and for
    smart_drafts_mode, on the full architecture with trained-like weights (two queries, ragged lengths)."""
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    cfg = ModelConfig(src_vocab_size=288, tgt_vocab_size=288, **PRODUCT_PREDICTION)
    sd = copy_task_state_dict(cfg, 77)
    src = synthetic_sources(3, 288, seed=4242, mean_len=40.0, std_len=12.0, min_len=12, max_len=80).to(dev)
    res = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("TTB_NO_FUSED_STATS", flag)
        eng = _engine(cfg, sd, "bf16")
        gen = TranslationInferenceBeamSearchSpeculative(eng, 120, n_best, 10, 7, 288, smart, 0, 1, 2, 7)
        res[flag] = (gen.generate(src).cpu().numpy(), gen.model_calls_num, gen.accepted_tokens_num, gen.gpu_launches)
        eng.close()
    (o_un, c_un, a_un, l_un), (o_fu, c_fu, a_fu, l_fu) = res["1"], res["0"]
    assert l_fu < l_un and c_fu == c_un and a_fu == a_un
    assert o_un.shape == o_fu.shape and np.array_equal(o_un[:, 0], o_fu[:, 0])
    assert (o_un == o_fu).all(-1).mean() >= 0.9
