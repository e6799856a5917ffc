#!/usr/bin/env python
"""Throughput of the sampling decoding (TranslationInferenceSampling, DESIGN.md section 15) against what it replaces and
against greedy decoding.

Full product-prediction architecture, bf16, trained-like copy weights (weights.copy_task_state_dict) and random weights,
--batches batches of --batch-size synthetic USPTO-MIT-shape sources.  Legs, timed with CUDA events after a warm-up of
every leg, alternating within every pass, median of --reps passes:
  * greedy      TranslationInferenceGreedy.generate (one prediction per source);
  * sample      S samples per source, top_k in {0, 5}, S in {1, 5, 10};
  * beam        the standard beam search with beam S (S in {5, 10}): today's way to get S predictions per source.
Rates are predictions (sample rows, beam hypotheses or greedy rows) per second.  A profiled pass per leg then reads the
`gemm_classifier` kernel-class time (the vocabulary projection with the arg-max or the draw fused into it; with the
fallback, the logits GEMM, and the `argmax` class holds sample_rows_kernel) per decoded row, for the greedy arg-max, the
fused draw and the forced fallback (TTB_NO_FUSED_ARGMAX=1).  One JSON line per weights kind, with the card name and power
limit read in the same run."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "scripts"))

from score import gpu_info  # noqa: E402
from translation_transformer_b200.decoding import (TranslationInferenceBeamSearch, TranslationInferenceGreedy,  # noqa: E402
                                                   TranslationInferenceSampling)
from translation_transformer_b200.model import B200Transformer  # noqa: E402
from translation_transformer_b200.synthetic import synthetic_sources  # noqa: E402
from translation_transformer_b200.weights import PRODUCT_PREDICTION, ModelConfig, copy_task_state_dict, random_init_state_dict  # noqa: E402

PAD, BOS, EOS, V = 0, 1, 2, 288
KC_GEMM_CLASSIFIER, KC_ARGMAX = 10, 11


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=8)
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5, help="timed passes (legs alternate within a pass)")
    ap.add_argument("--max-len", type=int, default=200)
    ap.add_argument("--weights", default="copy,random")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_sample.py needs a B200; there is no CPU path"
    dev = torch.device("cuda", 0)
    info = gpu_info(0)
    cfg = ModelConfig(src_vocab_size=V, tgt_vocab_size=V, **PRODUCT_PREDICTION)
    srcs = [synthetic_sources(args.batch_size, V, seed=900 + i).to(dev) for i in range(args.batches)]
    n_src = args.batches * args.batch_size
    L = args.max_len
    for kind in args.weights.split(","):
        sd = copy_task_state_dict(cfg, 1234) if kind == "copy" else random_init_state_dict(cfg, 1234)
        eng = B200Transformer(cfg, sd, precision="bf16", device=0)
        legs = {"greedy": (TranslationInferenceGreedy(eng, L, PAD, BOS, EOS), 1)}
        for S in (1, 5, 10):
            for k in (0, 5):
                legs[f"sample_S{S}_k{k}"] = (TranslationInferenceSampling(eng, L, S, PAD, BOS, EOS, temperature=1.0, top_k=k, seed=7), S)
        for S in (5, 10):
            legs[f"beam_{S}"] = (TranslationInferenceBeamSearch(eng, S, L, PAD, BOS, EOS), S)
        for gen, _ in legs.values():   # warm-up: every shape, graph and kernel of every leg
            for s in srcs:
                gen.generate(s)
        times = {name: [] for name in legs}
        steps = {}
        for _ in range(args.reps):
            for name, (gen, _) in legs.items():
                calls0 = gen.model_calls_num
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for s in srcs:
                    gen.generate(s)
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / 1e3)
                steps[name] = (gen.model_calls_num - calls0) / args.batches
        med = {name: statistics.median(t) for name, t in times.items()}
        rates = {name: round(n_src * legs[name][1] / med[name], 1) for name in legs}
        # classifier kernel-class time per decoded row: greedy arg-max, fused draw, forced fallback draw
        lib = eng.lib
        n_cls = lib.ttb_kernel_class_count()
        prof = {}
        for name, env in (("greedy_argmax", None), ("sample_S5_k0_fused", None), ("sample_S5_k5_fused", None),
                          ("sample_S5_k0_fallback", "1"), ("sample_S5_k5_fallback", "1")):
            leg = "greedy" if name.startswith("greedy") else name.rsplit("_", 1)[0]
            gen = legs[leg][0]
            if env:
                os.environ["TTB_NO_FUSED_ARGMAX"] = env
            lib.ttb_engine_set_profiling(eng._h, (1 << KC_GEMM_CLASSIFIER) | (1 << KC_ARGMAX))
            rows = 0
            for s in srcs:
                gen.generate(s)
                st = gen.last_stats
                rows += st.produced_tokens if leg != "greedy" else st.model_calls * s.shape[0]
            ms = (C.c_double * n_cls)()
            nl = (C.c_int64 * n_cls)()
            lib.ttb_engine_get_profile(eng._h, n_cls, ms, nl)
            lib.ttb_engine_set_profiling(eng._h, 0)
            os.environ.pop("TTB_NO_FUSED_ARGMAX", None)
            prof[name] = {"rows": rows, "gemm_classifier_ns_per_row": round(1e6 * ms[KC_GEMM_CLASSIFIER] / max(rows, 1), 2),
                          "argmax_class_ns_per_row": round(1e6 * ms[KC_ARGMAX] / max(rows, 1), 2),
                          "gemm_classifier_launches": int(nl[KC_GEMM_CLASSIFIER]), "argmax_class_launches": int(nl[KC_ARGMAX])}
        line = json.dumps({"weights": kind, "sources": n_src, "batch_size": args.batch_size, "max_len": L, "precision": "bf16",
                           "predictions_per_s": rates, "steps_per_batch": {k: round(v, 1) for k, v in steps.items()},
                           "median_s": {k: round(v, 4) for k, v in med.items()},
                           "spread_s": {k: [round(min(t), 4), round(max(t), 4)] for k, t in times.items()},
                           "classifier_profile": prof, **info})
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                print(line, file=f)
        eng.close()


if __name__ == "__main__":
    main()
