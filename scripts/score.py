#!/usr/bin/env python
"""Score the gold targets of a test set: the log-likelihood the model gives every target, teacher-forced, on ONE GPU.

    python scripts/score.py --src-file tests/golden/product_prediction_src_test.txt \\
                            --tgt-file tests/golden/product_prediction_tgt_test.txt --batch-size 4 --output out/scores.csv

Sources and targets are read, tokenised and batched as scripts/predict.py does (same options for the data and the model).
--output gets one CSV line per query, in file order, without a header: `index,n_tokens,logp` (scored tokens of the target,
EOS included, and the sum of their log-probabilities).  One JSON line on stdout: query count, scored tokens, mean negative
log-likelihood per token, perplexity, seconds of the scoring loop, GPU name and power limit.  Single GPU only: the test
set is scored on cuda:0."""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "scripts"))

from predict import load_batches, load_weights  # noqa: E402
from translation_transformer_b200.model import B200Transformer  # noqa: E402
from translation_transformer_b200.scoring import TranslationScorer  # noqa: E402
from translation_transformer_b200.weights import PRODUCT_PREDICTION, ModelConfig, random_init_state_dict  # noqa: E402


def parse(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--src-file", required=True)
    ap.add_argument("--tgt-file", required=True)
    ap.add_argument("--vocab-path", help="reference vocab.json (index -> token); built from the files when absent")
    ap.add_argument("--ckpt", help="torch file with the reference checkpoint (state_dict under 'state_dict', keys 'model.*')")
    ap.add_argument("--weights", default="random", choices=["random", "copy"],
                    help="without --ckpt: plain random init, or the trained-like copy circuit of weights.copy_task_state_dict")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--output", help="CSV of the per-query scores; omitted -> only the summary line is printed")
    ap.set_defaults(synthetic=0)
    return ap.parse_args(argv)


def gpu_info(device: int = 0) -> dict:
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power}


def main():
    args = parse()
    assert torch.cuda.is_available(), "score.py needs a B200; there is no CPU path"
    dev = torch.device("cuda", 0)
    tk, batches = load_batches(args)
    cfg = ModelConfig(src_vocab_size=tk.n_tokens, tgt_vocab_size=tk.n_tokens, src_pad_token_idx=tk.pad_token_idx,
                      tgt_pad_token_idx=tk.pad_token_idx, **PRODUCT_PREDICTION)
    sd = load_weights(args, tk)
    model = B200Transformer(cfg, sd if sd is not None else random_init_state_dict(cfg, args.seed), precision=args.precision, device=0)
    scorer = TranslationScorer(model, tk.pad_token_idx, tk.eos_token_idx)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    results = [scorer.score(b["src_tokens"].to(dev), b["tgt_tokens"].to(dev)) for b in batches]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    logp = torch.cat([r.logp for r in results]).double().cpu()
    ntok = torch.cat([r.n_tokens for r in results]).long().cpu()
    if args.output:
        Path(args.output).parent.mkdir(parents=True, exist_ok=True)
        with open(args.output, "w") as f:
            for i, (n, lp) in enumerate(zip(ntok.tolist(), logp.tolist())):
                f.write(f"{i},{n},{lp:.6f}\n")
    tokens = int(ntok.sum())
    nll = -float(logp.sum()) / max(tokens, 1)
    print(json.dumps({"queries": len(logp), "tokens": tokens, "mean_nll_per_token": round(nll, 6), "perplexity": round(math.exp(nll), 4),
                      "seconds": round(dt, 4), "precision": args.precision, "batch_size": args.batch_size, "weights": args.weights if not args.ckpt else "ckpt",
                      **gpu_info(), "output": args.output}), flush=True)
    model.close()


if __name__ == "__main__":
    main()
