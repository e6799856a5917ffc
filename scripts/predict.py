#!/usr/bin/env python
"""`main.py predict` for the hot path: decode a test set through the Lightning-shaped model and write the
reference's prediction CSV (BASELINE.json configs[4]: 40k-query test set sharded over the GPUs of one box).

    python scripts/predict.py --synthetic 40000 --generation greedy_speculative --batch-size 32 --output out/pred.csv
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 scripts/predict.py --synthetic 40000 ...
    python scripts/predict.py --src-file tests/golden/product_prediction_src_test.txt \
                              --tgt-file tests/golden/product_prediction_tgt_test.txt --batch-size 1

Mirrors what the reference does for `predict` (main.py -> Seq2SeqDM.predict_dataloader -> predict_step ->
PredictionWriter, seq2seq_wrappers.py:122-128,168-175; lightning_model.py:236-239; callbacks.py:42-64): fixed-size
batches in file order, right-padded with PAD.  Under torchrun the batches are drawn by all ranks and in-flight engines from
one shared queue (`--sharding dynamic`, default; `static` = contiguous shards), the predictions are all-gathered over NCCL
once at the end and rank 0 writes the CSV in file order: byte-identical to the one-GPU sequential run.  Without a
checkpoint the weights are random-init of the configured architecture (there are no checkpoints offline)."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

import torch
from torch.nn.utils.rnn import pad_sequence

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

from translation_transformer_b200.callbacks import PredictionWriter  # noqa: E402
from translation_transformer_b200.data_handling import ChemSMILESTokenizer  # noqa: E402
from translation_transformer_b200.distributed import gather_predictions, shard_batches  # noqa: E402
from translation_transformer_b200.synthetic import synthetic_sources  # noqa: E402
from translation_transformer_b200.weights import PRODUCT_PREDICTION  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--src-file")
    ap.add_argument("--tgt-file")
    ap.add_argument("--vocab-path", help="reference vocab.json (index -> token); built from the files when absent")
    ap.add_argument("--synthetic", type=int, default=0, help="decode this many synthetic USPTO-MIT-shape queries instead of a file")
    ap.add_argument("--vocab", type=int, default=288, help="vocabulary size of the synthetic queries")
    ap.add_argument("--ckpt", help="torch file with the reference checkpoint (state_dict under 'state_dict', keys 'model.*')")
    ap.add_argument("--generation", default="greedy_speculative",
                    choices=["greedy", "beam_search", "greedy_speculative", "beam_search_speculative", "sampling"])
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--beam-size", type=int, default=5)
    ap.add_argument("--max-len", type=int, default=200)
    ap.add_argument("--draft-len", type=int, default=10)
    ap.add_argument("--n-drafts", type=int, default=23)
    ap.add_argument("--smart-drafts-mode", action="store_true")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--seed", type=int, default=1234, help="seed of the random weights (without --ckpt)")
    ap.add_argument("--n-samples", type=int, default=5, help="--generation sampling: samples per source (CSV prediction_1..n)")
    ap.add_argument("--temperature", type=float, default=1.0, help="--generation sampling: soft-max temperature")
    ap.add_argument("--top-k", type=int, default=0, help="--generation sampling: draw from the k most likely tokens (0: all)")
    ap.add_argument("--sampling-seed", type=int, default=0,
                    help="--generation sampling: seed of the noise (a query's samples depend on its tokens and this seed only)")
    ap.add_argument("--output", help="prediction CSV (reference format); omitted -> predictions are not saved")
    ap.add_argument("--report-file")
    ap.add_argument("--in-flight", type=int, default=3,
                    help="batches decoded concurrently per GPU (one engine each, pipeline.py); 1 = the reference's sequential loop")
    ap.add_argument("--weights", default="random", choices=["random", "copy"],
                    help="without --ckpt: plain random init, or the trained-like copy circuit of weights.copy_task_state_dict "
                         "(queries finish at their own length: ragged finish times, real token sequences in the CSV)")
    ap.add_argument("--sharding", default="dynamic", choices=["dynamic", "static"],
                    help="dynamic: one queue of batch indices shared by all ranks and in-flight engines; static: contiguous shards per rank")
    return ap.parse_args()


def synthetic_tokenizer(vocab: int) -> ChemSMILESTokenizer:
    """Vocabulary of `vocab` entries: service tokens, then 'c' (the replace token the speculative loops ask for) and
    bracket atoms that the SMILES pattern splits back one to one."""
    tk = ChemSMILESTokenizer()
    enc = dict(tk.encoder_dict)
    for name in ["C", "O", "N", "c", "(", ")", "=", "1", "2", "n", ".", "F", "Cl", "Br", "S", "#"]:
        enc[name] = len(enc)
    while len(enc) < vocab:
        enc[f"[X{len(enc)}]"] = len(enc)
    tk.assign_vocab(enc)
    return tk


def load_batches(args):
    """-> tokenizer, list of {"src_tokens", "tgt_tokens"} batches in file order (CPU tensors)."""
    if args.synthetic:
        tk = synthetic_tokenizer(args.vocab)
        batches = []
        for i, lo in enumerate(range(0, args.synthetic, args.batch_size)):
            n = min(args.batch_size, args.synthetic - lo)
            src = synthetic_sources(n, args.vocab, seed=100003 + i)
            batches.append({"src_tokens": src, "tgt_tokens": src[:, :2].clone()})
        return tk, batches
    assert args.src_file, "--src-file or --synthetic is required"
    src_lines = [l.strip() for l in open(args.src_file) if l.strip()]
    tgt_lines = [l.strip() for l in open(args.tgt_file)] if args.tgt_file else [""] * len(src_lines)
    tgt_lines = [l for l in tgt_lines if l] if args.tgt_file else tgt_lines
    assert len(src_lines) == len(tgt_lines), "The source and target data have different lengths"
    tk = ChemSMILESTokenizer()
    if args.vocab_path:
        tk.load_vocab(args.vocab_path)
    else:
        tk.train_tokenizer(src_lines + tgt_lines)
    s = [torch.tensor(tk.encode(l)).long() for l in src_lines]
    t = [torch.tensor(tk.encode(l)).long() for l in tgt_lines]
    batches = []
    for lo in range(0, len(s), args.batch_size):
        batches.append({"src_tokens": pad_sequence(s[lo:lo + args.batch_size], batch_first=True, padding_value=tk.pad_token_idx),
                        "tgt_tokens": pad_sequence(t[lo:lo + args.batch_size], batch_first=True, padding_value=tk.pad_token_idx)})
    return tk, batches


def load_weights(args, tk):
    """State dict of --ckpt, the trained-like weights of --weights copy, or None (random init from --seed)."""
    if args.ckpt:
        sd = torch.load(args.ckpt, map_location="cpu", weights_only=True)
        sd = sd.get("state_dict", sd)
        return {k[len("model."):] if k.startswith("model.") else k: v for k, v in sd.items() if "positional_encoding" not in k}
    if args.weights == "copy":
        from translation_transformer_b200.weights import ModelConfig, copy_task_state_dict
        return copy_task_state_dict(ModelConfig(src_vocab_size=tk.n_tokens, tgt_vocab_size=tk.n_tokens, **PRODUCT_PREDICTION), args.seed)
    return None


def main_dynamic(args, model, tk, batches, n_best, rank, world, dev):
    """One queue of batch indices shared by all ranks and in-flight engines (distributed.BatchQueue) instead of contiguous
    static shards: a rank that drew long queries draws fewer batches.  Predictions are collected with ONE indexed all-gather
    at the end and written in file order, so the CSV is byte-identical to a one-GPU sequential run."""
    import torch.distributed as dist
    from translation_transformer_b200.distributed import BatchQueue, gather_indexed_predictions
    failures = []
    queue = BatchQueue(len(batches))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    model.on_predict_start()
    t0 = time.perf_counter()
    done = model.predict_queue(batches, queue, on_error=lambda i, ex: failures.append(i))
    fixed = []
    for i, pred in done:
        k = batches[i]["src_tokens"].shape[0]
        if pred is None:               # the reference's own failure modes (INTEGRATION.md §3): keep the row count
            pred = torch.zeros(k, n_best, args.max_len, dtype=torch.int64, device=dev)
        if pred.shape[2] < args.max_len:   # beam searches return the width they reached
            pred = torch.nn.functional.pad(pred, (0, args.max_len - pred.shape[2]))
        pred = pred[:, :, :args.max_len]
        if k < args.batch_size:        # the last batch of the file: same shape for the gather
            pred = torch.nn.functional.pad(pred, (0, 0, 0, 0, 0, args.batch_size - k))
        fixed.append((i, pred.contiguous()))
    everything = gather_indexed_predictions([i for i, _ in fixed], [p for _, p in fixed], len(batches), device=dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = time.perf_counter() - t0
    mine_n = torch.tensor([len(done)], dtype=torch.int64, device=dev)
    per_rank = [torch.zeros_like(mine_n) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, mine_n)
    else:
        per_rank = [mine_n]
    if rank == 0:
        model.on_predict_end()
        n = sum(b["src_tokens"].shape[0] for b in batches)
        if args.output:
            w = PredictionWriter(args.output)
            for i, b in enumerate(batches):
                w.write(tk, everything[i][:b["src_tokens"].shape[0]].cpu(), b)
        print(json.dumps({"queries": n, "n_gpus": world, "seconds": round(dt, 3), "smiles_per_s": round(n / dt, 1), "sharding": "dynamic queue",
                          "batches_per_rank": [int(x.item()) for x in per_rank], "generation": args.generation, "batch_size": args.batch_size,
                          "precision": args.precision, "batches_in_flight": max(1, args.in_flight), "weights": args.weights,
                          "model_calls_rank0": model._counter("model_calls_num"), "reference_failures_rank0": len(failures), "output": args.output}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import torch.distributed as dist
    from translation_transformer_b200.lightning_model import VanillaEncoderDecoderTransformerLightning
    assert torch.cuda.is_available(), "predict.py needs a B200; there is no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # NCCL logs (version banner) off stdout
        dist.init_process_group("nccl", device_id=dev)

    tk, batches = load_batches(args)
    sd = load_weights(args, tk)
    model = VanillaEncoderDecoderTransformerLightning(
        src_tokenizer=tk, tgt_tokenizer=tk, generation=args.generation, beam_size=args.beam_size,
        max_len=args.max_len, n_drafts=args.n_drafts, draft_len=args.draft_len, smart_drafts_mode=args.smart_drafts_mode,
        report_prediction_time=rank == 0, report_prediction_file=args.report_file, state_dict=sd, precision=args.precision,
        device=local_rank, seed=args.seed, batches_in_flight=max(1, args.in_flight), n_samples=args.n_samples,
        temperature=args.temperature, top_k=args.top_k, sampling_seed=args.sampling_seed, **PRODUCT_PREDICTION)

    mine = shard_batches(len(batches), rank, world)
    n_best = 1 if args.generation in ("greedy", "greedy_speculative") else (args.n_samples if args.generation == "sampling" else args.beam_size)
    if args.sharding == "dynamic":
        return main_dynamic(args, model, tk, batches, n_best, rank, world, dev)
    failures = 0
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    model.on_predict_start()
    t0 = time.perf_counter()
    local = []
    mine = list(mine)

    def failed(i, ex):               # the reference's own failure modes (INTEGRATION.md §3): keep the row count
        nonlocal failures
        failures += 1
        return torch.zeros(batches[mine[i]]["src_tokens"].shape[0], n_best, args.max_len, dtype=torch.int64, device=dev)

    if args.in_flight > 1:
        preds = model.predict_batches([batches[bi] for bi in mine], on_error=failed)
    else:
        def sequential():
            for i, bi in enumerate(mine):
                try:
                    yield model.predict_step({"src_tokens": batches[bi]["src_tokens"].to(dev, non_blocking=True)}, bi)
                except RuntimeError as ex:
                    yield failed(i, ex)
        preds = sequential()
    for pred in preds:
        if pred.shape[2] < args.max_len:   # beam searches return the width they reached
            pred = torch.nn.functional.pad(pred, (0, args.max_len - pred.shape[2]))
        local.append(pred[:, :, :args.max_len])
    local = torch.cat(local, dim=0) if local else torch.zeros(0, n_best, args.max_len, dtype=torch.int64, device=dev)
    counts = [sum(batches[b]["src_tokens"].shape[0] for b in shard_batches(len(batches), r, world)) for r in range(world)]
    allp = gather_predictions(local, counts=counts)     # NCCL all-gather, rank order == file order
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = time.perf_counter() - t0
    if rank == 0:
        model.on_predict_end()
        n = sum(counts)
        if args.output:
            w = PredictionWriter(args.output)
            lo = 0
            for b in batches:
                k = b["src_tokens"].shape[0]
                w.write(tk, allp[lo:lo + k].cpu(), b)
                lo += k
        print(json.dumps({"queries": n, "n_gpus": world, "seconds": round(dt, 3), "smiles_per_s": round(n / dt, 1),
                          "generation": args.generation, "batch_size": args.batch_size, "precision": args.precision,
                          "batches_in_flight": max(1, args.in_flight), "model_calls_rank0": model._counter("model_calls_num"), "reference_failures_rank0": failures,
                          "output": args.output}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
