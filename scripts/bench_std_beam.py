#!/usr/bin/env python
"""Timing of the standard (non-speculative) decoding strategies (standard_decoding.py) on synthetic sources, trained-like weights:
beam search, plain greedy for reference."""
import json
import os
import sys
import time
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
from translation_transformer_b200.decoding import TranslationInferenceBeamSearch, TranslationInferenceGreedy  # noqa: E402
from translation_transformer_b200.model import B200Transformer  # noqa: E402
from translation_transformer_b200.synthetic import synthetic_sources  # noqa: E402
from translation_transformer_b200.weights import ModelConfig, PRODUCT_PREDICTION, copy_task_state_dict  # noqa: E402


def main():
    bs, beam, steps = int(os.environ.get("BS", 8)), int(os.environ.get("BEAM", 5)), 4
    cfg = ModelConfig(src_vocab_size=288, tgt_vocab_size=288, **PRODUCT_PREDICTION)
    sd = copy_task_state_dict(cfg, 1234)
    dev = torch.device("cuda", 0)
    eng = B200Transformer(cfg, sd, precision="bf16", device=0)
    outs = {}
    for name, gen in (("beam_search", TranslationInferenceBeamSearch(eng, beam, 200, 0, 1, 2)), ("greedy", TranslationInferenceGreedy(eng, 200, 0, 1, 2))):
        srcs = [synthetic_sources(bs, 288, seed=500 + i).to(dev) for i in range(steps + 1)]
        gen.generate(srcs[0])
        torch.cuda.synchronize()
        c0, t0 = gen.model_calls_num, time.perf_counter()
        for s in srcs[1:]:
            out = gen.generate(s)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        outs[name] = out.cpu()
        print(json.dumps({"strategy": name, "bs": bs, "beam": beam if name == "beam_search" else 1, "smiles_per_s": round(bs * steps / dt, 1),
                          "ms_per_batch": round(1000 * dt / steps, 2), "decoder_calls_per_batch": (gen.model_calls_num - c0) / steps,
                          "top1_checksum": int(outs[name][:, 0].sum())}), flush=True)


if __name__ == "__main__":
    main()
