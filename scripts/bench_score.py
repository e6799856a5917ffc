#!/usr/bin/env python
"""Throughput of teacher-forced scoring (TranslationScorer, DESIGN.md section 14) against the route available without it:
`model(src.repeat_interleave(K, 0), tgt[:, :-1])` on the same engine, then torch `log_softmax` + `gather` + the same
scored-range mask.

Full product-prediction architecture, trained-like copy weights (weights.copy_task_state_dict), bf16, synthetic
USPTO-MIT-shape sources in batches of 32.  The K candidates of every source are the engine's own standard beam search
(beam K) on it, so candidate lengths and EOS positions are those of real n-best lists.  Both routes are timed with CUDA
events after a warm-up, alternating within the same run; their results are checked against each other first (scored
token counts equal, sums within the bf16 logit tolerance times the token count).  Prints one JSON line per K with the
card name and power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "scripts"))

from score import gpu_info  # noqa: E402
from translation_transformer_b200.decoding import TranslationInferenceBeamSearch  # noqa: E402
from translation_transformer_b200.model import B200Transformer  # noqa: E402
from translation_transformer_b200.scoring import TranslationScorer  # noqa: E402
from translation_transformer_b200.synthetic import synthetic_sources  # noqa: E402
from translation_transformer_b200.weights import PRODUCT_PREDICTION, ModelConfig, copy_task_state_dict  # noqa: E402

PAD, BOS, EOS, V = 0, 1, 2, 288


def forward_route(model, src, tgt, with_logits=False):
    """Scores of (B, K, W) candidates through the forward pass: encoder and cross-attention K/V once per candidate."""
    B, K, W = tgt.shape
    flat = tgt.reshape(B * K, W)
    logits = model(src.repeat_interleave(K, 0), flat[:, :-1])
    lp = torch.log_softmax(logits, dim=-1).gather(-1, flat[:, 1:, None])[..., 0]
    body = flat[:, 1:]
    stop = (body == PAD) | (body == EOS)
    seen = stop.int().cumsum(dim=1)
    scored = (seen == 0) | ((seen == 1) & (body == EOS))
    logp = torch.where(scored, lp, torch.zeros((), device=lp.device)).sum(dim=1).view(B, K)
    n = scored.sum(dim=1).view(B, K)
    return (logp, n, logits) if with_logits else (logp, n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=8, help="batches of --batch-size sources per timed pass")
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--reps", type=int, default=7, help="timed passes per route (alternating)")
    ap.add_argument("--ks", default="1,5,10")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_score.py needs a B200; there is no CPU path"
    dev = torch.device("cuda", 0)
    info = gpu_info(0)
    cfg = ModelConfig(src_vocab_size=V, tgt_vocab_size=V, **PRODUCT_PREDICTION)
    eng = B200Transformer(cfg, copy_task_state_dict(cfg, 1234), precision="bf16", device=0)
    scorer = TranslationScorer(eng, PAD, EOS)
    srcs = [synthetic_sources(args.batch_size, V, seed=700 + i).to(dev) for i in range(args.batches)]
    for K in [int(k) for k in args.ks.split(",")]:
        beam = TranslationInferenceBeamSearch(eng, K, 200, PAD, BOS, EOS)
        cands = [beam.generate(s) for s in srcs]
        # agreement of the two routes on every batch (also the warm-up of every shape)
        worst, n_tok = 0.0, 0
        for s, c in zip(srcs, cands):
            a = scorer.score(s, c)
            logp, n, logits = forward_route(eng, s, c, with_logits=True)
            assert torch.equal(a.n_tokens.long(), n), "scored token counts differ between the routes"
            tol = 2 * max(1.5e-2, 1e-2 * float(logits.abs().max()))
            err = ((a.logp - logp).abs() / (tol * n.clamp(min=1))).max().item()
            worst, n_tok = max(worst, err), n_tok + int(n.sum())
            assert err <= 1.0, f"routes disagree beyond the bf16 tolerance ({err:.3f} of it)"
        routes = {"scorer": lambda s, c: scorer.score(s, c), "forward": lambda s, c: forward_route(eng, s, c)}
        times = {name: [] for name in routes}
        for _ in range(args.reps):
            for name, fn in routes.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for s, c in zip(srcs, cands):
                    fn(s, c)
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / 1e3)
        n_cand = args.batches * args.batch_size * K
        med = {name: statistics.median(t) for name, t in times.items()}
        print(json.dumps({"K": K, "candidates": n_cand, "mean_candidate_width": round(sum(c.shape[2] for c in cands) / len(cands), 1),
                          "scored_tokens": n_tok,
                          "scorer_candidates_per_s": round(n_cand / med["scorer"], 1), "forward_candidates_per_s": round(n_cand / med["forward"], 1),
                          "speedup": round(med["forward"] / med["scorer"], 3),
                          "scorer_ms": [round(1e3 * t, 2) for t in times["scorer"]], "forward_ms": [round(1e3 * t, 2) for t in times["forward"]],
                          "max_err_of_bf16_tolerance": float(f"{worst:.3g}"), **info}), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
