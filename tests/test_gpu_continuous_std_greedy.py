"""Continuous batching of the standard greedy decoding (generate_batches): every batch's tokens and counters are
bit-identical to generate() on that batch alone, whatever the admission timing and the step counts of its neighbours."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from helpers import case_weights, load_json, load_npz
from test_gpu_continuous_beam import _bench_batches, _bench_model, _engine, _history
from translation_transformer_b200.synthetic import synthetic_sources
from translation_transformer_b200.weights import PRODUCT_PREDICTION

pytestmark = pytest.mark.gpu

PAD, BOS, EOS = 0, 1, 2


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _greedy(eng, max_len):
    from translation_transformer_b200.decoding import TranslationInferenceGreedy
    return TranslationInferenceGreedy(eng, max_len, PAD, BOS, EOS)


def _counters(g):
    return (g.model_calls_num, g.given_tokens)


def _one_by_one(make_gen, batches, calls=None):
    """generate() per batch on one generator: results and counters; `calls` (a list) receives each batch's model calls."""
    g = make_gen()
    res = []
    for b in batches:
        before = g.model_calls_num
        res.append(g.generate(b))
        if calls is not None:
            calls.append(g.model_calls_num - before)
    return res, _counters(g)


def _continuous(make_gen, batches, slots):
    g = make_gen()
    res = g.generate_batches(batches, slots=slots)
    return res, _counters(g)


def _assert_same(a, b):
    (ra, ca), (rb, cb) = a, b
    assert len(ra) == len(rb)
    for i, (x, y) in enumerate(zip(ra, rb)):
        assert x.shape == y.shape and torch.equal(x, y), f"batch {i} differs"
    assert ca == cb


# ---- 1. reference goldens (fp32), each case between filler batches, admission mid-loop ---------------------------------
@pytest.mark.parametrize("case", [c for c in load_json("standard_decoding.json") if c["kind"] == "greedy"], ids=lambda c: c["id"])
def test_goldens_between_fillers_fp32(dev, case):
    z = load_npz("standard_decoding.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    B, Ls = src.shape
    make = lambda: _greedy(eng, case["max_len"])
    # two fillers of B + 1 queries fill the slots; the case is admitted once one of them stops, the third filler behind it
    fill_a = synthetic_sources(B + 1, case["vocab"], seed=7 + B, mean_len=max(9, Ls - 4), std_len=4, min_len=8).to(dev)
    fill_c = synthetic_sources(B + 1, case["vocab"], seed=5 + B, mean_len=Ls + 12, std_len=4, min_len=8).to(dev)
    fill_b = synthetic_sources(B + 2, case["vocab"], seed=11 + B, mean_len=max(9, Ls - 2), std_len=5, min_len=8).to(dev)
    batches = [fill_a, fill_c, src, fill_b]
    slots = 2 * B + 2
    got = _continuous(make, batches, slots)
    _assert_same(_one_by_one(make, batches), got)
    assert max(_history(eng)) <= slots
    assert np.array_equal(got[0][2].cpu().numpy(), z[case["id"] + "_out"].astype(np.int64))
    g = make()
    g.generate_batches([src], slots=slots)
    assert g.model_calls_num == case["model_calls"] and g.given_tokens == case["given_tokens"]
    eng.close()


# ---- 2. bench shape (bf16): product-prediction model, mixed batch sizes ------------------------------------------------
@pytest.mark.parametrize("weights", ["copy", "random"])
def test_bench_shape_bf16_bit_identical(dev, weights):
    cfg, sd = _bench_model(PRODUCT_PREDICTION, weights)
    eng = _engine(cfg, sd, "bf16")
    sizes = (32, 32, 17, 32, 5, 32)
    batches = _bench_batches(dev, sizes, {}, 100003)
    bmax = max(sizes)
    # random weights drive every batch to max_len (a short one keeps the run short)
    max_len = 200 if weights == "copy" else 60
    make = lambda: _greedy(eng, max_len)
    ref = _one_by_one(make, batches)
    for slots in (bmax, 2 * bmax + 1, 4 * bmax, 16 * bmax):
        _assert_same(ref, _continuous(make, batches, slots))
        assert max(_history(eng)) <= slots
    eng.close()


# ---- 3. the slots of stopped batches are refilled while earlier batches still decode ----------------------------------
def test_refill_happens_and_slots_bound_the_live_count(dev):
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (32,) * 6, {}, 100003)
    make = lambda: _greedy(eng, 200)
    calls = []
    ref = _one_by_one(make, batches, calls)
    _assert_same(ref, _continuous(make, batches, 80))
    h = _history(eng)
    # more live slots than one batch holds, never more than the slots; batches overlap, so the loop takes fewer steps
    assert 32 < max(h) <= 80 and len(h) < sum(calls), (max(h), len(h), calls)
    _assert_same(ref, _continuous(make, batches, 32))
    h = _history(eng)
    assert max(h) <= 32 and len(h) == sum(calls)
    eng.close()


# ---- 4. edge cases: one-token sources, a single step, single-query batches, a batch that stops at once -----------------
def test_one_token_sources_and_single_query_batches(dev):
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (1, 4, 1, 1, 3, 1), {}, 100003)
    batches.insert(2, torch.full((2, 1), BOS, dtype=torch.int64, device=dev))   # generate() accepts Ls = 1
    make = lambda: _greedy(eng, 40)
    _assert_same(_one_by_one(make, batches), _continuous(make, batches, 6))
    _assert_same(_one_by_one(make, batches[:4]), _continuous(make, batches[:4], 4))
    eng.close()


def test_max_len_two_is_a_single_step(dev):
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (8, 5, 8, 3), {}, 100003)
    make = lambda: _greedy(eng, 2)
    calls = []
    ref = _one_by_one(make, batches, calls)
    assert calls == [1] * 4
    _assert_same(ref, _continuous(make, batches, 13))
    eng.close()


def test_batch_stopping_at_once_next_to_one_running_to_max_len(dev):
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    max_len = 30
    make = lambda: _greedy(eng, max_len)
    # the copy model predicts the source's next token: sources that end right behind BOS make every row predict EOS (or
    # PAD) in the first step; long sources keep every row busy until the rows are full
    short = [torch.tensor([[BOS, EOS] + [PAD] * k] * 3, dtype=torch.int64, device=dev) for k in (0, 1, 4)]
    calls = []
    _one_by_one(make, short, calls)
    first = next(s for s, c in zip(short, calls) if c == 1)
    long_a, long_b = (synthetic_sources(n, 288, seed=300007 + n, mean_len=80.0, std_len=5.0, min_len=60).to(dev) for n in (4, 2))
    batches = [long_a, first, long_b, first]
    calls = []
    ref = _one_by_one(make, batches, calls)
    assert calls == [max_len - 1, 1, max_len - 1, 1], calls
    # long_a and the first short batch fill the slots; long_b takes the short batch's slots while long_a decodes
    _assert_same(ref, _continuous(make, batches, 7))
    h = _history(eng)
    assert h[0] == 7 and max(h) <= 7 and len(h) < sum(calls), h
    eng.close()


# ---- 5. generate(), both continuous loops and back on one engine -------------------------------------------------------
def test_mode_switching_keeps_results(dev):
    from translation_transformer_b200.decoding import TranslationInferenceGreedySpeculative
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    batches = _bench_batches(dev, (32, 9, 17), {}, 100003)
    spec = lambda eng: TranslationInferenceGreedySpeculative(eng, 200, 10, 23, PAD, BOS, EOS, 3)

    def fresh(fn):
        eng = _engine(cfg, sd, "bf16")
        out = fn(eng)
        eng.close()
        return out

    want_single = fresh(lambda eng: [_greedy(eng, 200).generate(b) for b in batches])
    want_cont = fresh(lambda eng: _greedy(eng, 200).generate_batches(batches, slots=41))
    want_spec = fresh(lambda eng: spec(eng).generate_batches(batches, slots=41))
    eng = _engine(cfg, sd, "bf16")
    g = _greedy(eng, 200)
    first = [g.generate(b) for b in batches]
    mid = g.generate_batches(batches, slots=41)
    last = [g.generate(b) for b in batches]
    sp = spec(eng).generate_batches(batches, slots=41)
    again = g.generate_batches(batches, slots=41)
    for i in range(len(batches)):
        assert torch.equal(want_single[i], want_cont[i])
        assert torch.equal(first[i], want_single[i]) and torch.equal(last[i], want_single[i])
        assert torch.equal(mid[i], want_cont[i]) and torch.equal(again[i], want_cont[i])
        assert torch.equal(sp[i], want_spec[i])
    eng.close()
