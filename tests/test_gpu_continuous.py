"""Continuous batching of the speculative greedy loop (generate_batches): every batch's result, counters and trace are
bit-identical to generate() on that batch alone, whatever the admission timing."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from helpers import FULL, case_weights, load_json, load_npz
from translation_transformer_b200.synthetic import synthetic_sources
from translation_transformer_b200.weights import ModelConfig, copy_task_state_dict, random_init_state_dict

pytestmark = pytest.mark.gpu

PAD, BOS, EOS = 0, 1, 2


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _engine(cfg, sd, precision):
    from translation_transformer_b200.model import B200Transformer
    return B200Transformer(cfg, sd, precision=precision, device=0)


def _history(eng):
    import ctypes as C
    buf = (C.c_int32 * 65536)()
    n = eng.lib.ttb_engine_get_history(eng._h, buf, len(buf))
    return list(buf[:n])


def _one_by_one(make_gen, batches):
    """generate() per batch on one generator: results (or the exception), counters, trace."""
    g = make_gen()
    res = []
    for b in batches:
        try:
            res.append(g.generate(b))
        except RuntimeError as e:
            res.append(e)
    return res, (g.model_calls_num, g.accepted_tokens_num, g.produced_tokens_num), g.trace


def _continuous(make_gen, batches, slots):
    g = make_gen()
    res = g.generate_batches(batches, slots=slots, on_error=lambda i, e: e)
    return res, (g.model_calls_num, g.accepted_tokens_num, g.produced_tokens_num), g.trace


def _assert_same(a, b):
    (ra, ca, ta), (rb, cb, tb) = a, b
    assert len(ra) == len(rb)
    for i, (x, y) in enumerate(zip(ra, rb)):
        if isinstance(x, Exception):
            assert isinstance(y, RuntimeError) and str(y) == str(x), (i, x, y)
        else:
            assert not isinstance(y, Exception), (i, y)
            assert x.shape == y.shape and torch.equal(x, y), f"batch {i} differs"
    assert ca == cb
    assert ta == tb


# ---- 1. reference goldens (fp32), each case between two filler batches, admission mid-loop ----------------------------
@pytest.mark.parametrize("case", load_json("greedy_speculative.json"), ids=lambda c: c["id"])
def test_goldens_between_fillers_fp32(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    z = load_npz("greedy_speculative.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    B = case["B"]
    fill_a = synthetic_sources(B + 2, case["vocab"], seed=7 + B, mean_len=src.shape[1] + 6, std_len=8, min_len=3).to(dev)
    fill_b = synthetic_sources(max(1, B - 1), case["vocab"], seed=11 + B, mean_len=max(4, src.shape[1] - 4), std_len=5, min_len=3).to(dev)
    batches = [fill_a, src, fill_b]
    slots = max(b.shape[0] for b in batches) + 1

    def make(trace=False):
        return lambda: TranslationInferenceGreedySpeculative(eng, case["max_len"], case["draft_len"], case["n_drafts"], PAD, BOS, EOS,
                                                             case["replace"], keep_trace=trace)

    ref = _one_by_one(make(), batches)
    got = _continuous(make(), batches, slots)
    _assert_same(ref, got)
    out = got[0][1]
    if case["error"] is None:
        assert np.array_equal(out.cpu().numpy(), z[case["id"] + "_out"].astype(np.int64))
        g = make()()
        g.generate_batches([src], slots=slots)
        assert g.model_calls_num == case["model_calls"]
    else:
        assert isinstance(out, RuntimeError)   # and the fillers are what generate() gives for them (_assert_same)
        with pytest.raises(RuntimeError):
            make()().generate_batches(batches, slots=slots)

    ref_t = _one_by_one(make(True), batches)
    got_t = _continuous(make(True), batches, slots)
    _assert_same(ref_t, got_t)
    # the case's own iterations inside the trace: behind those of the first filler
    n0 = len(_one_by_one(make(True), [fill_a])[2])
    n1 = len(_one_by_one(make(True), [src])[2])
    trace = got_t[2][n0:n0 + n1]
    nacc = np.array([a for t in trace for a in t["n_accepted"]], dtype=np.int64)
    pick = np.array([p for t in trace for p in t["draft_index"]], dtype=np.int64)
    ref_nacc = z[case["id"] + "_nacc"].reshape(-1, case["n_drafts"])
    ref_pick = z[case["id"] + "_pick"]
    n = len(pick)
    assert n <= len(ref_pick) and (case["error"] is not None or n == len(ref_pick))
    assert np.array_equal(pick, ref_pick[:n])
    assert np.array_equal(nacc, ref_nacc[np.arange(n), ref_pick[:n]])
    eng.close()


# ---- 2. bench-shaped model, bf16, copy and random weights, graph path and traced (eager) path --------------------------
def _bench_model(weights):
    cfg = ModelConfig(src_vocab_size=288, tgt_vocab_size=288, **FULL)
    if weights == "copy":
        sd = copy_task_state_dict(cfg, 1234)
    else:
        sd = {k: v.clone() for k, v in random_init_state_dict(cfg, 1234).items()}
        sd["tgt_token_featurizer.embedding.weight"] = sd["src_token_featurizer.embedding.weight"]
    return cfg, sd


def _bench_batches(dev, sizes=(32, 32, 17, 32, 5, 32)):
    return [synthetic_sources(32, 288, seed=100003 + j)[:bs].to(dev) for j, bs in enumerate(sizes)]


@pytest.mark.parametrize("weights", ["copy", "random"])
def test_bench_shape_bf16_bit_identical(dev, weights):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    cfg, sd = _bench_model(weights)
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev)
    for trace in (False, True):
        make = lambda: TranslationInferenceGreedySpeculative(eng, 200, 10, 23, PAD, BOS, EOS, 3, keep_trace=trace)
        ref = _one_by_one(make, batches)
        for slots in (32, 48, 64, 200):
            _assert_same(ref, _continuous(make, batches, slots))
    eng.close()


# ---- 3. the slots of retired queries are refilled while earlier batches still decode ----------------------------------
def test_refill_happens_and_slots_bound_the_live_count(dev):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    cfg, sd = _bench_model("copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (32, 32, 32, 32))
    g = TranslationInferenceGreedySpeculative(eng, 200, 10, 23, PAD, BOS, EOS, 3)
    g.generate_batches(batches, slots=48)
    h = _history(eng)
    assert max(h) > 32 and max(h) <= 48, max(h)
    g.generate_batches(batches, slots=32)
    assert max(_history(eng)) <= 32
    eng.close()


# ---- 4. generate() -> generate_batches() -> generate() on one engine ---------------------------------------------------
def test_mode_switching_keeps_results(dev):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    cfg, sd = _bench_model("copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (32, 9))
    g = TranslationInferenceGreedySpeculative(eng, 200, 10, 23, PAD, BOS, EOS, 3)
    first = [g.generate(b) for b in batches]
    mid = g.generate_batches(batches, slots=40)
    last = [g.generate(b) for b in batches]
    again = g.generate_batches(batches, slots=40)
    for a, b, c, d in zip(first, mid, last, again):
        assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(a, d)
    eng.close()
