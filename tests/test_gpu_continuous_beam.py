"""Continuous batching of the speculative beam search (generate_batches): every batch's hypotheses, counters and trace are
bit-identical to generate() on that batch alone, whatever the admission timing and the draft lengths of its neighbours."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from helpers import case_weights, load_json, load_npz
from translation_transformer_b200.synthetic import synthetic_sources
from translation_transformer_b200.weights import PRODUCT_PREDICTION, SINGLE_STEP_RETRO, ModelConfig, copy_task_state_dict, random_init_state_dict

pytestmark = pytest.mark.gpu

PAD, BOS, EOS, REPLACE = 0, 1, 2, 3


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


def _draft_history(eng):
    """(draft length of every decoder call, smallest draft length of the batches in it) of the last continuous loop."""
    import ctypes as C
    a, b = (C.c_int32 * 65536)(), (C.c_int32 * 65536)()
    n = eng.lib.ttb_engine_get_draft_history(eng._h, a, b, 65536)
    return list(a[:n]), list(b[:n])


def _counters(g):
    return (g.model_calls_num, g.accepted_tokens_num, g.produced_non_pad_tokens, g.n_drafts)


def _one_by_one(make_gen, batches, calls=None):
    """generate() per batch on one generator: results (or the exception), counters, trace; `calls` (a list) receives
    each batch's model calls."""
    g = make_gen()
    res = []
    for b in batches:
        before = g.model_calls_num
        try:
            res.append(g.generate(b))
        except (RuntimeError, AssertionError) as e:
            res.append(e)
        if calls is not None:
            calls.append(g.model_calls_num - before)
    return res, _counters(g), g.trace


def _schedule(sizes, calls, slots):
    """The admission rule of the continuous loop (whole batches, list order, between iterations) replayed on the host:
    slots in use per iteration and each batch's first iteration."""
    used, nxt, it, h, start, open_ = 0, 0, 0, [], [], []
    while True:
        for j in [j for j in open_ if start[j] + calls[j] == it]:
            open_.remove(j)
            used -= sizes[j]
        while nxt < len(sizes) and slots - used >= sizes[nxt]:
            start.append(it)
            open_.append(nxt)
            used += sizes[nxt]
            nxt += 1
        if used == 0:
            return h, start
        h.append(used)
        it += 1


def _joins_mid_flight(j, calls, start):
    """batch j is admitted while a batch admitted before it is still decoding"""
    return any(start[i] < start[j] < start[i] + calls[i] for i in range(len(start)) if i != j)


def _continuous(make_gen, batches, slots):
    g = make_gen()
    res = g.generate_batches(batches, slots=slots, on_error=lambda i, e: e)
    return res, _counters(g), g.trace


def _same_trace(ta, tb):
    assert len(ta) == len(tb)
    for x, y in zip(ta, tb):
        assert np.array_equal(x["n_accepted"], y["n_accepted"]) and np.array_equal(x["pick"], y["pick"])


def _assert_same(a, b):
    (ra, ca, ta), (rb, cb, tb) = a, b
    assert len(ra) == len(rb)
    for i, (x, y) in enumerate(zip(ra, rb)):
        if isinstance(x, Exception):
            assert type(y) is type(x) and str(y) == str(x), (i, x, y)
        else:
            assert not isinstance(y, Exception), (i, y)
            assert x.shape == y.shape and torch.equal(x, y), f"batch {i} differs"
    assert ca == cb
    _same_trace(ta, tb)


# ---- 1. reference goldens (fp32), each case between two filler batches, admission mid-loop ----------------------------
def _cases():
    return [("beam_speculative", False, c) for c in load_json("beam_speculative.json")] + \
           [("beam_smart", True, c) for c in load_json("beam_smart.json")]


@pytest.mark.parametrize("kind,smart,case", _cases(), ids=lambda v: v["id"] if isinstance(v, dict) else str(v))
def test_goldens_between_fillers_fp32(dev, kind, smart, case):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    z = load_npz(kind + ".npz")
    cfg, sd = case_weights(case)
    eng = _engine(cfg, sd, "fp32")
    src = torch.from_numpy(z[case["id"] + "_src"].astype(np.int64)).to(dev)
    B, Ls = src.shape

    def make(trace=False):
        return lambda: TranslationInferenceBeamSearchSpeculative(eng, case["max_len"], case["n_best"], case["draft_len"], case["n_drafts"],
                                                                 case["vocab"], smart, PAD, BOS, EOS, case["C_token"], keep_trace=trace)

    # two fillers of B + 1 queries start together and fill the slots; the case is admitted when the first of them stops.
    # Fillers that take different numbers of iterations are picked from a few candidates, so that the other one is still
    # decoding then (with weights under which every batch runs to max_len no such pair exists: the case then follows them).
    cands = [synthetic_sources(B + 1, case["vocab"], seed=sd_ + B, mean_len=m, std_len=4, min_len=8).to(dev)
             for sd_, m in ((7, max(9, Ls - 4)), (5, Ls + 12), (13, 9), (17, Ls + 24))]
    n_calls = []
    _one_by_one(make(), cands, n_calls)
    i, j = next(((i, j) for i in range(len(cands)) for j in range(i + 1, len(cands)) if n_calls[i] != n_calls[j]), (0, 1))
    if n_calls[i] > n_calls[j]:
        i, j = j, i
    fill_a, fill_c = cands[i], cands[j]   # the shorter one first
    fill_b = synthetic_sources(B + 2, case["vocab"], seed=11 + B, mean_len=max(9, Ls - 2), std_len=5, min_len=8).to(dev)
    batches = [fill_a, fill_c, src, fill_b]
    slots = 2 * B + 2

    calls = []
    ref = _one_by_one(make(), batches, calls)
    h, start = _schedule([b.shape[0] for b in batches], calls, slots)
    if calls[0] != calls[1]:
        assert _joins_mid_flight(2, calls, start), (calls, start)
    got = _continuous(make(), batches, slots)
    _assert_same(ref, got)
    assert _history(eng) == h
    _assert_same(_one_by_one(make(True), batches), _continuous(make(True), batches, slots))
    out = got[0][2]
    if case["error"] is None:
        assert np.array_equal(out.cpu().numpy(), z[case["id"] + "_out"].astype(np.int64))
        g = make()()
        g.generate_batches([src], slots=slots)
        assert g.model_calls_num == case["model_calls"]
    else:
        assert isinstance(out, AssertionError)   # and the fillers are what generate() gives for them (_assert_same)
        assert not any(isinstance(got[0][j], Exception) for j in (0, 1, 3))
        with pytest.raises(AssertionError):
            make()().generate_batches(batches, slots=slots)
    eng.close()


# ---- 2. bench shapes (bf16): configs[2] in both draft modes, configs[3] (n_best 10, unfused statistics) ----------------
def _bench_model(arch, weights):
    cfg = ModelConfig(src_vocab_size=288, tgt_vocab_size=288, **arch)
    if weights == "copy":
        sd = copy_task_state_dict(cfg, 1234)
    else:
        sd = {k: v.clone() for k, v in random_init_state_dict(cfg, 1234).items()}
        sd["tgt_token_featurizer.embedding.weight"] = sd["src_token_featurizer.embedding.weight"]
    return cfg, sd


WORKLOADS = {
    # arch, n_best, n_drafts, smart, batch sizes (mixed), source shape
    "beam": (PRODUCT_PREDICTION, 5, 23, False, (4, 4, 2, 4, 3, 4, 1, 4), {}),
    "beam_smart": (PRODUCT_PREDICTION, 5, 23, True, (4, 3, 4, 1, 4, 2), {}),
    "retro": (SINGLE_STEP_RETRO, 10, 2, False, (8, 5, 8, 8, 3, 8), dict(mean_len=45.0, std_len=15.0, min_len=12, max_len=150)),
}


def _bench_batches(dev, sizes, src_kw, seed):
    return [synthetic_sources(max(sizes), 288, seed=seed + j, **src_kw)[:bs].to(dev) for j, bs in enumerate(sizes)]


@pytest.mark.parametrize("weights", ["copy", "random"])
@pytest.mark.parametrize("workload", list(WORKLOADS))
def test_bench_shape_bf16_bit_identical(dev, workload, weights):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    arch, n_best, n_drafts, smart, sizes, src_kw = WORKLOADS[workload]
    cfg, sd = _bench_model(arch, weights)
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, sizes, src_kw, 300007)
    bmax = max(sizes)
    # random weights drive every batch to max_len (a short one keeps the run short)
    max_len = 200 if weights == "copy" else 60
    for trace in (False, True):
        make = lambda: TranslationInferenceBeamSearchSpeculative(eng, max_len, n_best, 10, n_drafts, 288, smart, PAD, BOS, EOS, REPLACE,
                                                                 keep_trace=trace)
        ref = _one_by_one(make, batches)
        for slots in ((bmax, 2 * bmax + 1, 4 * bmax) if not trace else (2 * bmax + 1,)):
            _assert_same(ref, _continuous(make, batches, slots))
    eng.close()


@pytest.mark.parametrize("workload", list(WORKLOADS))
def test_batches_below_the_call_draft_length_bf16(dev, workload, monkeypatch):
    """A batch whose draft length has dropped near max_len shares decoder calls that run at a larger one; its positions
    must come out as in generate() at its own draft length.  TTB_BEAM_CB_FULL_DL=1 runs every call at the full draft
    length, so that every batch's last iterations are such iterations; without it they occur where batches of different
    progress overlap."""
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    arch, n_best, n_drafts, smart, sizes, src_kw = WORKLOADS[workload]
    cfg, sd = _bench_model(arch, "random")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, sizes, src_kw, 300007)
    make = lambda: TranslationInferenceBeamSearchSpeculative(eng, 60, n_best, 10, n_drafts, 288, smart, PAD, BOS, EOS, REPLACE, keep_trace=True)
    ref = _one_by_one(make, batches)
    slots = 2 * max(sizes) + 1
    for full in (False, True):
        monkeypatch.setenv("TTB_BEAM_CB_FULL_DL", "1" if full else "0")
        _assert_same(ref, _continuous(make, batches, slots))
        call_dl, min_dl = _draft_history(eng)
        assert len(call_dl) == len(_history(eng)) and all(b <= a for a, b in zip(call_dl, min_dl))
        if full:   # iterations in which a batch ran below the call's draft length did happen
            assert any(b < a for a, b in zip(call_dl, min_dl)), (call_dl, min_dl)
    eng.close()


# ---- 3. the slots of finished batches are refilled while earlier batches still decode ---------------------------------
def test_refill_happens_and_slots_bound_the_live_count(dev):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (4,) * 8, {}, 100003)
    calls = []
    _one_by_one(lambda: TranslationInferenceBeamSearchSpeculative(eng, 200, 5, 10, 23, 288, False, PAD, BOS, EOS, REPLACE), batches, calls)
    g = TranslationInferenceBeamSearchSpeculative(eng, 200, 5, 10, 23, 288, False, PAD, BOS, EOS, REPLACE)
    g.generate_batches(batches, slots=10)
    h = _history(eng)
    sched, start = _schedule([4] * 8, calls, 10)
    assert h == sched and max(h) <= 10
    # at least one batch is admitted into slots freed while a batch admitted before it is still decoding
    assert any(_joins_mid_flight(j, calls, start) for j in range(2, 8)), (calls, start)
    g.generate_batches(batches, slots=4)
    assert max(_history(eng)) <= 4
    eng.close()


# ---- 4. generate() -> generate_batches() -> generate() -> generate_batches() on one engine ----------------------------
def test_mode_switching_keeps_results(dev):
    from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative
    cfg, sd = _bench_model(PRODUCT_PREDICTION, "copy")
    eng = _engine(cfg, sd, "bf16")
    batches = _bench_batches(dev, (4, 3, 4), {}, 100003)
    g = TranslationInferenceBeamSearchSpeculative(eng, 200, 5, 10, 23, 288, False, PAD, BOS, EOS, REPLACE)
    first = [g.generate(b) for b in batches]
    mid = g.generate_batches(batches, slots=9)
    last = [g.generate(b) for b in batches]
    again = g.generate_batches(batches, slots=9)
    for a, b, c, d in zip(first, mid, last, again):
        assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(a, d)
    eng.close()
