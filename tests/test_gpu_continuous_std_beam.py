"""Continuous batching of the standard beam search (generate_batches): every batch's hypotheses and counters are
bit-identical to generate() on that batch alone, whatever the admission timing and the widths of its neighbours."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from helpers import case_weights, load_json, load_npz
from test_gpu_continuous_beam import _bench_batches, _bench_model, _engine, _history, _joins_mid_flight, _schedule
from translation_transformer_b200.synthetic import synthetic_sources
from translation_transformer_b200.weights import PRODUCT_PREDICTION, SINGLE_STEP_RETRO

pytestmark = pytest.mark.gpu

PAD, BOS, EOS = 0, 1, 2


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


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


# ---- 1. reference goldens (fp32), each case between two filler batches, admission mid-loop ----------------------------
@pytest.mark.parametrize("case", [c for c in load_json("standard_decoding.json") if c["kind"] == "beam"], ids=lambda c: c["id"])
def test_goldens_between_fillers_fp32(dev, case):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    z = load_npz("standard_decoding.npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    B, Ls = src.shape
    make = lambda: TranslationInferenceBeamSearch(eng, case["beam_size"], case["max_len"], PAD, BOS, EOS)

    # two fillers of B + 1 queries start together and fill the slots; the case is admitted when the first of them stops.
    # Fillers that take different numbers of steps are picked from a few candidates, so that the other one is still
    # decoding then (with weights under which every batch runs to max_len no such pair exists: the case then follows them).
    cands = [synthetic_sources(B + 1, case["vocab"], seed=sd_ + B, mean_len=m, std_len=4, min_len=8).to(dev)
             for sd_, m in ((7, max(9, Ls - 4)), (5, Ls + 12), (13, 9), (17, Ls + 24), (19, 12), (23, Ls), (29, 10), (31, Ls + 6),
                            (37, 20), (41, Ls + 40))]
    n_calls = []
    _one_by_one(make, cands, n_calls)
    i, j = next(((i, j) for i in range(len(cands)) for j in range(i + 1, len(cands)) if n_calls[i] != n_calls[j]), (0, 1))
    if n_calls[i] > n_calls[j]:
        i, j = j, i
    fill_a, fill_c = cands[i], cands[j]   # the shorter one first
    fill_b = synthetic_sources(B + 2, case["vocab"], seed=11 + B, mean_len=max(9, Ls - 2), std_len=5, min_len=8).to(dev)
    batches = [fill_a, fill_c, src, fill_b]
    slots = 2 * B + 2

    calls = []
    ref = _one_by_one(make, batches, calls)
    h, start = _schedule([b.shape[0] for b in batches], calls, slots)
    if calls[0] != calls[1]:
        assert _joins_mid_flight(2, calls, start), (calls, start)
    else:   # admissions then only happen at multiples of one batch's step count: no batch can join mid-flight
        assert len(set(n_calls)) == 1, n_calls
    got = _continuous(make, batches, slots)
    _assert_same(ref, got)
    assert _history(eng) == h
    out = got[0][2]
    assert np.array_equal(out.cpu().numpy(), z[case["id"] + "_out"].astype(np.int64))
    g = make()
    g.generate_batches([src], slots=slots)
    assert g.model_calls_num == case["model_calls"] and g.given_tokens == case["given_tokens"]
    eng.close()


# ---- 2. bench shapes (bf16): product prediction with beam 5, 6+6 retrosynthesis with beam 10 ---------------------------
WORKLOADS = {
    # arch, beam size, batch sizes (mixed), source shape
    "product_beam5": (PRODUCT_PREDICTION, 5, (8, 8, 3, 8, 5, 8, 1, 8), {}),
    "retro_beam10": (SINGLE_STEP_RETRO, 10, (8, 5, 8, 8, 3, 8), dict(mean_len=45.0, std_len=15.0, min_len=12, max_len=150)),
}


@pytest.mark.parametrize("weights", ["copy", "random"])
@pytest.mark.parametrize("workload", list(WORKLOADS))
def test_bench_shape_bf16_bit_identical(dev, workload, weights):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    arch, beam, sizes, src_kw = WORKLOADS[workload]
    cfg, sd = _bench_model(arch, weights)
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, sizes, src_kw, 300007)
    bmax = max(sizes)
    # random weights drive every batch to max_len (a short one keeps the run short)
    max_len = 200 if weights == "copy" else 60
    make = lambda: TranslationInferenceBeamSearch(eng, beam, max_len, PAD, BOS, EOS)
    ref = _one_by_one(make, batches)
    for slots in (bmax, 2 * bmax + 1, 4 * bmax, 16 * bmax):
        _assert_same(ref, _continuous(make, batches, slots))
        assert max(_history(eng)) <= slots
    eng.close()


# ---- 3. the slots of stopped batches are refilled while earlier batches still decode ----------------------------------
def test_refill_happens_and_history_matches_the_schedule(dev):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (4,) * 8, {}, 100003)
    make = lambda: TranslationInferenceBeamSearch(eng, 5, 200, PAD, BOS, EOS)
    calls = []
    ref = _one_by_one(make, batches, calls)
    got = _continuous(make, batches, 10)
    _assert_same(ref, got)
    h = _history(eng)
    sched, start = _schedule([4] * 8, calls, 10)
    assert h == sched and max(h) <= 10
    # at least one batch is admitted into slots freed while a batch admitted before it is still decoding
    assert any(_joins_mid_flight(j, calls, start) for j in range(2, 8)), (calls, start)
    eng.close()


# ---- 4. a batch of one-token sources (generate() accepts Ls = 1) ----------------------------------------------------------
def test_single_token_sources(dev):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (4, 3), {}, 100003) + [torch.full((2, 1), BOS, dtype=torch.int64, device=dev)]
    make = lambda: TranslationInferenceBeamSearch(eng, 5, 40, PAD, BOS, EOS)
    _assert_same(_one_by_one(make, batches), _continuous(make, batches, 6))
    eng.close()


# ---- 5. generate() -> generate_batches() -> generate() on one engine ---------------------------------------------------
def test_mode_switching_keeps_results(dev):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearch
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    batches = _bench_batches(dev, (4, 3, 4), {}, 100003)

    def fresh(fn):
        eng = _engine(cfg, sd, "bf16")
        out = fn(TranslationInferenceBeamSearch(eng, 5, 200, PAD, BOS, EOS))
        eng.close()
        return out

    want_single = fresh(lambda g: [g.generate(b) for b in batches])
    want_cont = fresh(lambda g: g.generate_batches(batches, slots=9))
    eng = _engine(cfg, sd, "bf16")
    g = TranslationInferenceBeamSearch(eng, 5, 200, PAD, BOS, EOS)
    first = [g.generate(b) for b in batches]
    mid = g.generate_batches(batches, slots=9)
    last = [g.generate(b) for b in batches]
    for a, b, c, w1, w2 in zip(first, mid, last, want_single, want_cont):
        assert torch.equal(a, w1) and torch.equal(c, w1) and torch.equal(b, w2) and torch.equal(w1, w2)
    eng.close()
