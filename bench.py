#!/usr/bin/env python
"""Benchmark of the hot path: the Molecular Transformer driven by the speculative decoding loops.

    python bench.py --gpus N --steps K --warmup W              our arm: libttb200 on B200 (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...    reference arm: the reference's own PyTorch code on the host cores

Workloads (`--workload`, BASELINE.json configs[1..3]); one "step" = one batch of synthetic queries decoded to completion
through the public generator classes (`TranslationInferenceGreedySpeculative.generate` / `...BeamSearchSpeculative.generate`):

    greedy  product prediction, greedy speculative, bs 32, draft_len 10, n_drafts 23, max_len 200        (configs[1], default)
    beam    product prediction, speculative beam search, bs 4, n_best 5, draft_len 10, n_drafts 23       (configs[2])
    retro   single-step retrosynthesis (6+6 layers), speculative beam search, bs 8, n_best 10, draft_len 10, n_drafts 2
            (configs[3]; scripts/single_step_retrosynthesis.sh:166-174), USPTO-50k-shape sources

Weights (`--weights`): `random` (default, what BASELINE.json's north_star names) = plain random init: nothing ever emits EOS,
every batch decodes all its queries to the width limit and the reference returns all-PAD rows -- the worst case and a
fixed amount of work per step; `copy` = the same random-init weights with the deterministic copy circuit of
`weights.copy_task_state_dict` laid over them, a stand-in for a TRAINED model (no checkpoints offline): predictions
follow the source, drafts are accepted at realistic rates, every query ends with EOS at its own length, so batches
retire query by query and the predictions are real token sequences.  The default line reports both (the second as
`trained_like`) and, on one GPU, the beam / retro workloads (trained-like weights) as `workloads`.

The timed batches are drawn from ONE queue shared by all ranks and in-flight engines (`distributed.BatchQueue`): nobody
owns a static shard.  `--scaling weak` (default) times N*K batches on N GPUs, `--scaling strong` a fixed set of
`--queries` queries whatever N is.  The side workloads of the default line time `--steps` batches each as well.  Every
GPU output is checked: against the reference goldens of the same batch (tests/golden/bench_configs.npz) and against the
reference run live on the host for a few queries (`parity`).  `--dump-outputs DIR` saves the prediction of each workload's
last timed step; the inputs depend only on the arguments, so two builds run with the same arguments compare file by file.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

from translation_transformer_b200.synthetic import synthetic_sources  # noqa: E402
from translation_transformer_b200.weights import (ModelConfig, PRODUCT_PREDICTION, SINGLE_STEP_RETRO, copy_task_state_dict,  # noqa: E402
                                                  random_init_state_dict)

PAD, BOS, EOS, REPLACE = 0, 1, 2, 7   # REPLACE plays the role of the "c" token (lightning_model.py:117)
RETRO_SRC = dict(mean_len=45.0, std_len=15.0, min_len=12, max_len=150)
WORKLOADS = {
    "greedy": dict(kind="greedy", arch="product", bs=32, draft_len=10, n_drafts=23, src_seed=100003, src_kw={}, draw=32,
                   golden={"copy": "cfg1_copy", "random": "cfg1_random"},
                   metric="SMILES/sec (greedy speculative, product prediction)",
                   name="product-prediction greedy speculative bs=32 draft_len=10 n_drafts=23 (BASELINE.json configs[1])"),
    "beam": dict(kind="beam", arch="product", bs=4, n_best=5, draft_len=10, n_drafts=23, src_seed=100003, src_kw={}, draw=32,
                 golden={"copy": "cfg2_copy"}, metric="SMILES/sec (beam-search speculative, product prediction)",
                 name="product-prediction speculative beam search bs=4 n_best=5 draft_len=10 n_drafts=23 (BASELINE.json configs[2])"),
    "retro": dict(kind="beam", arch="retro", bs=8, n_best=10, draft_len=10, n_drafts=2, src_seed=200003, src_kw=RETRO_SRC, draw=8,
                  golden={"copy": "cfg3_copy"}, metric="SMILES/sec (beam-search speculative, single-step retrosynthesis)",
                  name="single-step retrosynthesis (6+6 layers) speculative beam search bs=8 n_best=10 draft_len=10 n_drafts=2 "
                       "(BASELINE.json configs[3]; scripts/single_step_retrosynthesis.sh:166-174)"),
}
ARCH = {"product": PRODUCT_PREDICTION, "retro": SINGLE_STEP_RETRO}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=18)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="greedy", choices=list(WORKLOADS))
    ap.add_argument("--weights", default="random", choices=["random", "copy"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--queries", type=int, default=4096, help="size of the fixed query set of --scaling strong")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--max-len", type=int, default=200)
    ap.add_argument("--vocab", type=int, default=288)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--cpu-queries", type=int, default=2, help="queries of the live CPU parity / baseline sample; --impl reference: > 2 fixes the per-step sample, otherwise it is sized to a ~3 minute run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-insitu", action="store_true", help="skip the extra CUPTI-profiled step (kernels_in_situ)")
    ap.add_argument("--no-extra-workloads", action="store_true", help="only the selected workload (no random-init / beam / retro side figures)")
    ap.add_argument("--tie-break", default="torch_cpu", choices=["torch_cpu", "lowest_index"])
    ap.add_argument("--in-flight", type=int, default=0,
                    help="batches decoded concurrently per GPU, one engine + stream each (translation_transformer_b200/pipeline.py); "
                         "1 = strictly one batch after the other, also always measured and reported as `one_batch_in_flight`; 0 (default) = 3 "
                         "for the random-init greedy workload (every batch keeps all its queries to the end), 8 for the trained-like greedy "
                         "workload whose batches thin out while they decode, 12 for the beam searches (measured: DESIGN.md section 4c)")
    ap.add_argument("--clock-period-ms", type=int, default=200, help="nvidia-smi sampling period; 0 disables the sampler")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the prediction of the last timed step of every measured workload to "
                         "DIR/<workload>_<weights>.npy (token ids as float32), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 1:
        ap.error("--steps and --warmup must be at least 1 (the warm-up batches size every workspace and feed the parity check)")
    return args


# ------------------------------------------------------------------------------------------------
class Workload:
    """One of WORKLOADS with a weight set: configuration, weights and the synthetic batches."""

    def __init__(self, key, weights, args):
        self.key, self.weights, self.args = key, weights, args
        self.w = WORKLOADS[key]
        self.kind, self.bs = self.w["kind"], self.w["bs"]
        self.cfg = ModelConfig(src_vocab_size=args.vocab, tgt_vocab_size=args.vocab, **ARCH[self.w["arch"]])
        if weights == "copy":
            self.sd = copy_task_state_dict(self.cfg, args.seed)
        else:
            self.sd = {k: v.clone() for k, v in random_init_state_dict(self.cfg, args.seed).items()}
            self.sd["tgt_token_featurizer.embedding.weight"] = self.sd["src_token_featurizer.embedding.weight"]
        self.out_width = args.max_len if self.kind == "greedy" else args.max_len + max(5, self.w["draft_len"]) + 4
        self.n_best = 1 if self.kind == "greedy" else self.w["n_best"]
        self.golden_id = self.w["golden"].get(weights) if (args.vocab, args.seed, args.max_len) == (288, 1234, 200) else None

    def batch(self, j):
        """Synthetic batch number j of the job (j = 0 is the batch the reference goldens were recorded on)."""
        return synthetic_sources(self.w["draw"], self.args.vocab, seed=self.w["src_seed"] + j, **self.w["src_kw"])[:self.bs]

    def describe(self):
        a = self.cfg
        wt = ("trained-like copy-circuit weights over random init (weights.copy_task_state_dict" if self.weights == "copy" else "random-init weights (")
        src = "USPTO-50k-shape sources (12..150 tokens, mean 45)" if self.w["arch"] == "retro" else "USPTO-MIT-shape sources (20..198 tokens, mean 80)"
        return (f"{self.w['name']}, max_len={self.args.max_len}; Molecular Transformer {a.embedding_dim}/{a.feedforward_dim}/"
                f"{a.num_encoder_layers}+{a.num_decoder_layers}/{a.num_heads}, {wt}, seed {self.args.seed}), vocab {self.args.vocab}; synthetic {src}")

    def generator(self, eng, keep_trace=False):
        from translation_transformer_b200.decoding import TranslationInferenceBeamSearchSpeculative, TranslationInferenceGreedySpeculative
        a, w = self.args, self.w
        if self.kind == "greedy":
            return TranslationInferenceGreedySpeculative(eng, a.max_len, w["draft_len"], w["n_drafts"], PAD, BOS, EOS, REPLACE,
                                                         tie_break=a.tie_break, keep_trace=keep_trace)
        return TranslationInferenceBeamSearchSpeculative(eng, a.max_len, w["n_best"], w["draft_len"], w["n_drafts"], a.vocab, False,
                                                         PAD, BOS, EOS, REPLACE, tie_break=a.tie_break, keep_trace=keep_trace)

    def pad_out(self, out):
        """(B, n_best, W) prediction -> fixed width (the beam search returns the width it reached)."""
        if out.shape[-1] == self.out_width:
            return out
        res = torch.zeros(out.shape[:-1] + (self.out_width,), dtype=out.dtype, device=out.device)
        res[..., :out.shape[-1]] = out
        return res

    # ---- the reference itself (oracle/_ref) or its port (oracle/), on `device` -----------------------------------
    def reference_generator(self, device="cpu"):
        from oracle import ref_runner
        a, w = self.args, self.w
        if ref_runner.available():
            m = ref_runner.build_model(self.cfg, self.sd, device)
            if self.kind == "greedy":
                return ref_runner.greedy_speculative(m, a.max_len, w["draft_len"], w["n_drafts"], PAD, BOS, EOS, REPLACE), "reference"
            return ref_runner.beam_speculative(m, a.max_len, w["n_best"], w["draft_len"], w["n_drafts"], a.vocab, False, PAD, BOS, EOS, REPLACE), "reference"
        assert device == "cpu", "the oracle port is a CPU restatement"
        from oracle.transformer import OracleTransformer
        m = OracleTransformer(self.sd, self.cfg.num_heads)
        if self.kind == "greedy":
            from oracle.greedy_speculative import GreedySpeculativeOracle
            return GreedySpeculativeOracle(m, a.max_len, w["draft_len"], w["n_drafts"], PAD, BOS, EOS, REPLACE), "port"
        from oracle.beam_speculative import BeamSearchSpeculativeOracle
        return BeamSearchSpeculativeOracle(m, a.max_len, w["n_best"], w["draft_len"], w["n_drafts"], a.vocab, False, PAD, BOS, EOS, REPLACE), "port"


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=200):
        self.index, self.proc, self.lines, self.period_ms = index, None, [], period_ms

    def start(self):
        if self.period_ms <= 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period_ms), "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "tflops_burst": d["bf16_tflops"],
                "source": "measured (MEASURED_PEAKS.json, sustained bf16)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_kernel_table():
    """Per-kernel counters of the committed `ncu --set full` capture (profiles/*_ncu_kernels.json, written by
    scripts/ncu_summary.py from the .ncu-rep): DRAM bytes per launch, tensor-pipe activity."""
    files = sorted((REPO / "profiles").glob("*_ncu_kernels.json"))
    if not files:
        return None, {}
    try:
        return files[-1].name, json.load(open(files[-1]))["kernels"]
    except Exception:
        return None, {}


def class_work(name, wl, cfg, hist, src_lens_mean, fused_ln=True, fused_ffn=True, chained_ffn=False, precision="bf16"):
    """Algorithmic (flops, bytes) of ALL launches of a kernel class over the greedy iterations in `hist` (live queries per
    iteration); per-unit figures are in DESIGN.md §4.  With the fused kernels the sub-layer tails (bias + residual +
    LayerNorm, fp32 and bf16 copies of the residual stream) are part of the GEMM classes and the whole feed-forward
    block is the class `gemm_ffn1`."""
    E, F, V, L = cfg.embedding_dim, cfg.feedforward_dim, cfg.tgt_vocab_size, cfg.num_decoder_layers
    D, N = wl["draft_len"], wl["n_drafts"]
    per_q = N * (D + 1)
    rows = sum(h * per_q for h in hist)           # token rows summed over iterations
    ab = 2 if precision == "bf16" else 4           # activation bytes
    n_it = len(hist)
    ln_flops = 8.0 * rows * E
    stream_bytes = rows * E * (4 + 4 + ab)          # residual in, residual out (fp32), low-precision copy out
    if name == "gemm_ffn1" and fused_ffn:
        f, b = (4.0 * rows * E * F + ln_flops) * L, (rows * E * ab + stream_bytes) * L + 2 * E * F * ab * L * n_it
        if chained_ffn:   # the launch also computes the cross-attention out-projection + LayerNorm (att in, x in/out fp32)
            f += (2.0 * rows * E * E + ln_flops) * L
            b += (rows * E * ab + rows * E * 8) * L + E * E * ab * L * n_it
        return f, b
    if name in ("gemm_self_out", "gemm_cross_out") and fused_ln:
        f = (2.0 * rows * E * E + ln_flops) * L
        if name == "gemm_self_out":
            f += 2.0 * rows * E * E * L               # chained cross-attention query projection
        return f, (rows * E * ab + stream_bytes) * L + E * E * ab * L * n_it
    if name == "gemm_ffn2" and fused_ln:
        return (2.0 * rows * E * F + ln_flops) * L, (rows * F * ab + stream_bytes) * L + E * F * ab * L * n_it
    gemm = {"gemm_qkv": (E, 3 * E, ab), "gemm_self_out": (E, E, 4), "gemm_cross_q": (E, E, ab), "gemm_cross_out": (E, E, 4),
            "gemm_ffn1": (E, F, ab), "gemm_ffn2": (F, E, 4)}
    if name in gemm:
        K, Nn, ob = gemm[name]
        return 2.0 * rows * K * Nn * L, (rows * K * ab + rows * Nn * ob) * L + K * Nn * ab * L * n_it
    if name == "gemm_classifier":
        return 2.0 * rows * E * V, rows * E * ab + rows * 4 + E * V * ab * n_it
    if name == "cross_attn":
        lk = src_lens_mean
        return 4.0 * rows * lk * E * L, (rows * E * ab * 2 + sum(hist) * lk * 2 * E * ab) * L
    if name == "self_attn":
        # keys: accepted prefix (grows while decoding) + causal half of the draft row
        flops = sum(4.0 * h * per_q * (it + 1 + (D + 2) / 2.0) * E for it, h in enumerate(hist)) * L
        byts = sum(h * (per_q * 4 * E * ab + (it + 1) * 2 * E * ab) for it, h in enumerate(hist)) * L
        return flops, byts
    if name == "add_layernorm":
        return 8.0 * rows * E * 3 * L, rows * E * (4 + 4 + 4 + ab) * 3 * L
    return 0.0, 0.0


def insitu_kernel_times(fn):
    """One extra step under CUPTI (torch.profiler): per kernel name the number of launches, the average duration and the
    average time between the end of the preceding kernel and its own end, i.e. what the kernel adds to the step inside
    the CUDA-graph / programmatic-dependent-launch pipeline (the event brackets of the instrumented step cannot see
    that: they serialise every launch)."""
    from collections import defaultdict
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = sorted(((e.time_range.start, e.time_range.end, e.name) for e in prof.events()
                 if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Mem")), key=lambda t: t[0])
    agg = defaultdict(lambda: [0, 0.0, 0.0])
    prev_end = None
    for st, en, name in ev:
        a = agg[name.split("(")[0].split("::")[-1].split("<")[0]]
        a[0] += 1
        a[1] += en - st
        a[2] += en - max(st, prev_end) if prev_end is not None and prev_end > st else en - st
        prev_end = en if prev_end is None else max(prev_end, en)
    return {k: {"launches": n, "avg_us": round(d / n, 2), "avg_added_us": round(g / n, 2)} for k, (n, d, g) in agg.items()}


CLASS_KERNEL = {"gemm_ffn1": ("ffn_pair_kernel", "ffn_fused_kernel"), "self_attn": ("attn_tc_kernel", "attn_mma_kernel"),
                "cross_attn": ("attn_tc_kernel", "attn_mma_kernel"),
                "gemm_qkv": ("gemm_pair_k256_kernel", "gemm_bf16_tc_persistent_kernel"), "gemm_self_out": ("gemm_resid_ln_kernel",),
                "gemm_cross_out": ("gemm_resid_ln_kernel",), "gemm_classifier": ("classifier_argmax_kernel",)}


# ------------------------------------------------------------------------------------------------
def compare_with_golden(wl, out):
    """GPU prediction of batch 0 against the UNMODIFIED reference's output for the same batch (committed fixture)."""
    if wl.golden_id is None or not (REPO / "tests/golden/bench_configs.npz").exists():
        return None
    z = np.load(REPO / "tests/golden/bench_configs.npz")
    if wl.golden_id + "_out" not in z.files:
        return None
    ref = z[wl.golden_id + "_out"].astype(np.int64)
    src = z[wl.golden_id + "_src"].astype(np.int64)
    if not np.array_equal(src, wl.batch(0).numpy()):
        return {"checked": False, "why": "the fixture's batch is not this run's batch 0"}
    o = out.cpu().numpy()
    W = max(o.shape[-1], ref.shape[-1])
    po = np.zeros(o.shape[:-1] + (W,), np.int64); po[..., :o.shape[-1]] = o
    pr = np.zeros(ref.shape[:-1] + (W,), np.int64); pr[..., :ref.shape[-1]] = ref
    same_top1 = (po[:, 0] == pr[:, 0]).all(-1)
    res = {"checked": True, "against": f"unmodified reference, tests/golden/bench_configs.npz:{wl.golden_id}", "queries": int(len(same_top1)),
           "top1_identical": int(same_top1.sum()), "non_pad_tokens_in_reference": int((pr != PAD).sum())}
    if wl.kind == "beam":
        res["hypotheses_identical"] = int((po == pr).all(-1).sum())
        res["hypotheses"] = int(po.shape[0] * po.shape[1])
    return res


def compare_trace_with_golden(wl, gen_traced, src_dev):
    """All-PAD predictions say nothing (random-init weights never finish), so the loop itself is compared: the accepted length
    and the chosen draft of every (iteration, live query) of a traced decode of batch 0 against what the unmodified reference
    did on the same batch (recorded through hooks, tests/golden/make_golden_bench.py).  fp32 engines reproduce every cell
    (tests/test_gpu_bench_configs.py); the bf16 engine follows the reference until the first near-tie of two logits flips."""
    if wl.kind != "greedy" or wl.golden_id is None or not (REPO / "tests/golden/bench_configs.npz").exists():
        return None
    z = np.load(REPO / "tests/golden/bench_configs.npz")
    if wl.golden_id + "_nacc" not in z.files:
        return None
    N = wl.w["n_drafts"]
    ref_nacc = z[wl.golden_id + "_nacc"].astype(np.int64).reshape(-1, N)
    ref_pick = z[wl.golden_id + "_pick"].astype(np.int64)
    ref_acc = ref_nacc[np.arange(len(ref_pick)), ref_pick]
    try:
        gen_traced.generate(src_dev)
    except RuntimeError:
        pass
    nacc = np.array([a for t in gen_traced.trace for a in t["n_accepted"]], dtype=np.int64)
    pick = np.array([p_ for t in gen_traced.trace for p_ in t["draft_index"]], dtype=np.int64)
    n = min(len(nacc), len(ref_acc))
    eq = (nacc[:n] == ref_acc[:n]) & (pick[:n] == ref_pick[:n])
    return {"cells": int(n), "reference_cells": int(len(ref_acc)), "cells_identical": int(eq.sum()),
            "first_differing_cell": int(np.argmax(~eq)) if (~eq).any() else int(n),
            "what": "(iteration, live query) cells of batch 0: accepted length and chosen draft index vs the unmodified reference"}


def compare_with_live_reference(wl, out, nq):
    """The reference (oracle/_ref, else the oracle port) decodes the first `nq` queries of batch 0 on the host now; the
    GPU rows for the same queries must carry the same tokens.  Returns (parity dict, cpu_baseline dict).  Greedy queries
    are independent of their batch mates; the beam search is run on the sub-batch by both sides."""
    gen, kind = wl.reference_generator("cpu")
    src = wl.batch(0)[:nq].clone()
    torch.set_num_threads(host_threads())
    t0 = time.perf_counter()
    err = None
    with torch.inference_mode():
        try:
            ref = gen.generate(src)
        except (RuntimeError, AssertionError) as ex:
            ref, err = None, str(ex)[:80]
    dt = time.perf_counter() - t0
    base = {"value": nq / dt, "unit": "SMILES/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"first {nq} queries of batch 0, full decode, {gen.model_calls_num} decoder calls, {dt:.1f} s"}
    if ref is None:
        return {"checked": False, "why": f"the reference raised: {err}"}, base
    o, r = out.cpu().numpy(), ref.cpu().numpy()
    W = max(o.shape[-1], r.shape[-1])
    po = np.zeros(o.shape[:-1] + (W,), np.int64); po[..., :o.shape[-1]] = o
    pr = np.zeros(r.shape[:-1] + (W,), np.int64); pr[..., :r.shape[-1]] = r
    same = (po[:, 0] == pr[:, 0]).all(-1)
    return {"checked": True, "against": f"{kind} run on the host in this process", "queries": int(nq), "top1_identical": int(same.sum()),
            "non_pad_tokens_in_reference": int((pr != PAD).sum())}, base


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation (oracle/_ref; the oracle port when that copy is absent) with
    all host threads.  Each step decodes a bounded sample (`--cpu-queries` queries) of the step's batch; plus, once, the
    same unmodified code on cuda:0 (`reference_gpu_eager`, context for "over the reference's PyTorch path")."""
    if rank != 0:
        return
    torch.set_num_threads(host_threads())   # torchrun exports OMP_NUM_THREADS=1 to its workers
    wl = Workload(args.workload, args.weights, args)
    gen, kind = wl.reference_generator("cpu")

    def decode(src):
        t0 = time.perf_counter()
        with torch.inference_mode():
            try:
                gen.generate(src)
            except (RuntimeError, AssertionError):
                pass
        return time.perf_counter() - t0

    # sample size: as many queries of the step's batch as keep the whole run within ~3 minutes (calibrated on 2 queries)
    t_cal = decode(wl.batch(0)[:min(2, wl.bs)]) / min(2, wl.bs)
    n_steps = args.warmup + args.steps
    nq = args.cpu_queries if args.cpu_queries > 0 else 0
    nq = max(1, min(wl.bs, nq if nq > 2 else int(180.0 / n_steps / max(t_cal, 1e-3))))
    times = [decode(wl.batch(i)[:nq]) for i in range(n_steps)][args.warmup:]
    total = sum(times)
    value = nq * len(times) / total
    line = {"impl": "reference", "metric": wl.w["metric"], "value": value, "unit": "SMILES/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * total / len(times),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl.describe(), "sample": f"{nq} of {wl.bs} queries per step"},
            "cpu_baseline": {"value": value, "unit": "SMILES/s", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": f"{nq} of {wl.bs} queries per step, {len(times)} steps, full decode (max_len {args.max_len})"},
            "e2e": {"value": value, "unit": "SMILES/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if nq < wl.bs and t_cal * wl.bs * 0.6 < 90.0:
        # one WHOLE batch as the reference's predict loop decodes it (batched GEMMs are cheaper per query than the sample's)
        dt = decode(wl.batch(args.warmup))
        line["full_batch"] = {"value": wl.bs / dt, "unit": "SMILES/s", "seconds": round(dt, 1), "batch_size": wl.bs,
                              "what": "batch `warmup` of the job decoded whole, once (same configuration as the GPU arm's step)"}
    if torch.cuda.is_available() and kind == "reference":
        try:   # informational: the reference's normal deployment is eager PyTorch on a GPU
            g2, _ = wl.reference_generator("cuda:0")
            with torch.inference_mode():
                g2.generate(wl.batch(0).cuda())
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                nb = 2
                for i in range(1, 1 + nb):
                    try:
                        g2.generate(wl.batch(i).cuda())
                    except (RuntimeError, AssertionError):
                        pass
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
            line["reference_gpu_eager"] = {"value": nb * wl.bs / dt, "unit": "SMILES/s", "batches": nb, "batch_size": wl.bs,
                                           "what": "the unmodified reference (oracle/_ref) in eager fp32 PyTorch on cuda:0, whole batches"}
        except Exception as ex:
            line["reference_gpu_eager"] = {"error": str(ex)[:120]}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class Runner:
    """Engines + generators of one workload on this rank, and the timed regions over a shared batch queue."""

    def __init__(self, wl, args, local_rank, world, n_fly):
        from translation_transformer_b200.model import B200Transformer
        from translation_transformer_b200.pipeline import InFlightDecoder
        self.wl, self.args, self.world, self.local_rank = wl, args, world, local_rank
        self.dev = torch.device("cuda", local_rank)
        self.engs = [B200Transformer(wl.cfg, wl.sd, precision=args.precision, device=local_rank) for _ in range(n_fly)]
        self.gens = [wl.generator(e) for e in self.engs]
        self.fly = InFlightDecoder(self.gens, device=local_rank)
        self.one = InFlightDecoder(self.gens[:1], device=local_rank)
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)   # > 126 MB L2
        self.errors = []
        self.cache = {}

    def host_batch(self, j):
        if j not in self.cache:
            self.cache[j] = self.wl.batch(j).pin_memory()
        return self.cache[j]

    def counters(self):
        names = ("model_calls_num", "gpu_launches", "accepted_tokens_num") + (("produced_tokens_num",) if self.wl.kind == "greedy" else ("produced_non_pad_tokens",))
        return [sum(getattr(g, n) for g in self.gens) for n in names]

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def decode_one(self, j):
        """Batch j on the first engine, synchronously (warm-up, parity)."""
        src = self.host_batch(j).to(self.dev, non_blocking=True)
        return self.gens[0].generate(src)

    def timed(self, first, n_batches, e2e, decoder=None, resident=None):
        """Decode batches first .. first+n_batches-1 of the job; every rank and every in-flight engine pulls the next index
        from one shared queue.  e2e: inputs start in pinned host memory, each prediction is copied back to pinned host
        memory inside the region.  Returns (ms as max over ranks, batches decoded by this rank, failed batches)."""
        import torch.distributed as dist
        from translation_transformer_b200.distributed import BatchQueue, gather_indexed_predictions
        decoder = decoder or self.fly
        wl = self.wl
        for j in range(first, first + n_batches):
            self.host_batch(j)
        if not e2e:
            resident = resident if resident is not None else {j: self.host_batch(j).to(self.dev) for j in range(first, first + n_batches)}
        out_hosts = {}
        if e2e:
            out_hosts = {j: torch.empty(wl.bs, wl.n_best, wl.out_width, dtype=torch.int64).pin_memory() for j in range(first, first + n_batches)}
        q = BatchQueue(n_batches)
        failed = []

        def next_item():
            i = q.next()
            return None if i is None else (first + i, first + i)

        tls = threading.local()

        def pre(j):
            tls.j = j
            self.flush.zero_()                                   # on the worker's stream, like everything of its step
            return self.host_batch(j).to(self.dev, non_blocking=True) if e2e else resident[j]

        def post(o):
            o = wl.pad_out(o)
            if e2e:                                              # device -> pinned host copy of the step's prediction, on the worker's stream
                out_hosts[tls.j].copy_(o, non_blocking=True)
            return o

        def on_error(j, ex):   # reference-faithful failure modes (oracle/greedy_speculative.py); not counted as throughput
            failed.append(j)
            self.errors.append(str(ex)[:80])
            return None

        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record()
        done = decoder.drain(next_item, pre=pre, post=post, on_error=on_error)
        good = [(j, o) for j, o in done if o is not None]
        # predictions of every rank collected once, in batch order (NCCL all-gather; identity on one GPU)
        gathered = gather_indexed_predictions([j - first for j, _ in good], [o for _, o in good], n_batches, device=self.dev)
        ev1.record()
        self.barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=self.dev)
        nfail = torch.tensor([len(failed)], device=self.dev, dtype=torch.int64)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(nfail)
        self.last_gathered = gathered
        return float(ms.item()), len(done), int(nfail.item())

    def close(self):
        self.fly.close()
        self.one.close()
        for e in self.engs:
            e.close()
        self.flush = None


def measure_workload(wl, args, local_rank, world, rank, n_fly, steps, warmup, n_timed_batches, full):
    """Warm-up, parity, timed regions (resident, end to end, strictly sequential) of one workload.  `full` adds the
    instrumented step (per-class CUDA events -> roofline) and the CUPTI in-situ step."""
    R = Runner(wl, args, local_rank, world, n_fly)
    res = {}
    # ---- warm-up (also sizes every workspace) + parity of batch 0 ---------------------------------------------------
    out0 = None
    for g_i, g in enumerate(R.gens):
        for i in range(warmup):
            try:
                o = g.generate(R.host_batch(i).to(R.dev))
                if g_i == 0 and i == 0:
                    out0 = o.clone()
            except RuntimeError as ex:
                R.errors.append(str(ex)[:80])
    if n_fly > 1:    # and W more through the worker threads, `n_fly` at a time (thread start-up, per-thread CUDA state)
        from translation_transformer_b200.distributed import BatchQueue
        q = BatchQueue(warmup * n_fly, local=True)
        R.fly.drain(lambda: (lambda i: None if i is None else (i, i % warmup))(q.next()), pre=lambda j: R.host_batch(j).to(R.dev),
                    on_error=lambda j, ex: None)
    if n_fly > 1 and world == 1:   # the worker thread of the strictly sequential decoder as well (its first job pays the thread's CUDA set-up)
        from translation_transformer_b200.distributed import BatchQueue
        q1 = BatchQueue(2, local=True)
        R.one.drain(lambda: (lambda i: None if i is None else (i, i % warmup))(q1.next()), pre=lambda j: R.host_batch(j).to(R.dev),
                    on_error=lambda j, ex: None)
    torch.cuda.synchronize()
    parity = {}
    if rank == 0 and out0 is not None:
        parity["golden"] = compare_with_golden(wl, out0)
        if parity["golden"] is not None and wl.kind == "greedy":
            parity["golden"]["trace"] = compare_trace_with_golden(wl, wl.generator(R.engs[0], keep_trace=True), R.host_batch(0).to(R.dev))
    res["_out0"] = out0
    first = warmup
    lib, eng, gen = R.engs[0].lib, R.engs[0], R.gens[0]
    shares, hist, n_cls, names = {}, [], 0, []
    if full and wl.kind == "greedy":
        # ---- one instrumented step: CUDA-event time of every kernel class -> dominant kernel ---------
        n_cls = lib.ttb_kernel_class_count()
        names = [lib.ttb_kernel_class_name(i).decode() for i in range(n_cls)]
        lib.ttb_engine_set_profiling(eng._h, (1 << n_cls) - 1)
        R.flush.zero_()
        try:
            gen.generate(R.host_batch(first).to(R.dev))
        except RuntimeError as ex:
            R.errors.append(str(ex)[:80])
        ms_arr, n_arr = (C.c_double * n_cls)(), (C.c_int64 * n_cls)()
        lib.ttb_engine_get_profile(eng._h, n_cls, ms_arr, n_arr)
        shares = {names[i]: {"ms": round(ms_arr[i], 3), "launches": int(n_arr[i])} for i in range(n_cls) if n_arr[i]}
        tot_ms = sum(v["ms"] for v in shares.values()) or 1.0
        for v in shares.values():
            v["share"] = round(v["ms"] / tot_ms, 4)
        buf = (C.c_int32 * (args.max_len + 2))()
        n_hist = lib.ttb_engine_get_history(eng._h, buf, args.max_len + 2)
        hist = list(buf[:n_hist])
        lib.ttb_engine_set_profiling(eng._h, 0)
    # ---- timed regions ----------------------------------------------------------------------------------------------
    if world > 1:   # untimed pass through the shared queue and the NCCL all-gather (the first collective of a kind sets up its channels)
        R.timed(0, world * n_fly, False)
    one_n = max(1, min(n_timed_batches, steps))
    one_ms, _, one_fail = R.timed(first, one_n, False, decoder=R.one) if (n_fly > 1 and world == 1) else (None, 0, 0)
    c0 = R.counters()
    sampler = ClockSampler(local_rank, args.clock_period_ms)
    if rank == 0 and full:
        sampler.start()
    ms, mine, nfail = R.timed(first, n_timed_batches, False)
    clocks = sampler.stop() if (rank == 0 and full) else None
    last = R.last_gathered[-1]          # None when the last batch ended in a reference failure mode
    res["last"] = None if last is None else last.cpu()
    c1 = R.counters()
    e2e_ms, _, e2e_fail = R.timed(first, n_timed_batches, True)
    insitu = None
    if full and rank == 0 and not args.no_insitu:
        try:
            src_d = R.host_batch(first).to(R.dev)
            insitu = insitu_kernel_times(lambda: gen.generate(src_d))   # rank-local: no collective in here
        except Exception as ex:   # CUPTI not available: the event-bracket figures stand alone
            insitu = {"error": str(ex)[:120]}
    delta = torch.tensor([b - a for a, b in zip(c0, c1)], dtype=torch.int64, device=R.dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(delta)
    calls, launches, accepted, produced = [int(x) for x in delta.tolist()]
    q_ok = (n_timed_batches - nfail) * wl.bs
    res.update({"value": q_ok / (ms / 1000.0), "ms": ms, "batches": n_timed_batches, "failed_batches": nfail, "batches_this_rank": mine,
                "e2e_value": (n_timed_batches - e2e_fail) * wl.bs / (e2e_ms / 1000.0), "e2e_ms": e2e_ms,
                "one_value": (one_n - one_fail) * wl.bs / (one_ms / 1000.0) if one_ms else None, "one_ms": one_ms, "one_batches": one_n,
                "calls": calls, "launches": launches, "accepted": accepted, "produced": produced, "clocks": clocks, "shares": shares,
                "hist": hist, "insitu": insitu, "parity": parity, "errors": R.errors[:3],
                "h2d": int(R.host_batch(first).numel() * 8), "d2h": int(wl.bs * wl.n_best * wl.out_width * 8),
                "src_len_mean": float((R.host_batch(first) != PAD).sum().item()) / wl.bs})
    R.close()
    return res


def roofline_tables(wl, args, m, peaks):
    """`roofline` (dominant class) and `roofline_all` (every decoder class) from the instrumented step of a greedy workload."""
    shares, hist, insitu = m["shares"], m["hist"], m["insitu"]
    if not shares or not hist:
        return None, None
    fused_ln = "add_layernorm" not in shares
    fused_ffn = "gemm_ffn2" not in shares
    chained_ffn = fused_ffn and "gemm_cross_out" not in shares
    ncu_file, ncu = ncu_kernel_table()
    balance = peaks["tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    table = {}
    for cls, sh in shares.items():
        if cls in ("encoder", "misc"):
            continue
        f, b = class_work(cls, wl.w, wl.cfg, hist, m["src_len_mean"], fused_ln, fused_ffn, chained_ffn, args.precision)
        n = max(sh["launches"], 1)
        us = 1000.0 * sh["ms"] / n
        tensor = f / max(b, 1.0) >= balance
        row = {"launches": sh["launches"], "share_of_step": sh["share"], "avg_us_event_bracket": round(us, 2),
               "flops_per_launch": f / n, "bytes_per_launch": b / n, "bound": "tensor" if tensor else "hbm"}
        per = (f if tensor else b) / n
        unit = 1e12 if tensor else 1e9
        peak = peaks["tflops"] if tensor else peaks["hbm_gbs"]
        row["frac_event_bracket"] = round(per / (us * 1e-6) / unit / peak, 4) if us > 0 else None
        k = next((kn for kn in CLASS_KERNEL.get(cls, ()) if insitu and kn in insitu), None) if insitu and "error" not in insitu else None
        # several classes can share one kernel name (self / cross attention; the two out-projections): in-situ figures are per name
        if k:
            row["kernel"] = k
            row["in_situ_us"] = insitu[k]["avg_added_us"]
            shared = [c for c in shares if k in CLASS_KERNEL.get(c, ())]
            if len(shared) == 1:
                row["frac_in_situ"] = round(per / (insitu[k]["avg_added_us"] * 1e-6) / unit / peak, 4)
        kn = next((kn for kn in CLASS_KERNEL.get(cls, ()) if kn in ncu), None)
        if kn:
            row["ncu"] = ncu[kn]
        table[cls] = row
    dominant = max(table, key=lambda c: shares[c]["ms"])
    d = table[dominant]
    tensor = d["bound"] == "tensor"
    per = d["flops_per_launch"] if tensor else d["bytes_per_launch"]
    ach = per / (d["avg_us_event_bracket"] * 1e-6) / (1e12 if tensor else 1e9)
    label = {"gemm_ffn1": ("ffn_pair_kernel (cross out-proj+LayerNorm2 + FFN1+ReLU+FFN2+residual+LayerNorm3, cta_group::2)" if chained_ffn else
                           "ffn_fused_kernel (FFN1+ReLU+FFN2+residual+LayerNorm)") if fused_ffn else "gemm_ffn1"}.get(dominant, d.get("kernel", dominant))
    traffic = d.get("ncu", {}).get("dram_bytes_per_launch")
    roof = {"bound": d["bound"], "achieved": ach, "peak": peaks["tflops"] if tensor else peaks["hbm_gbs"], "unit": "TFLOP/s" if tensor else "GB/s",
            "frac": ach / (peaks["tflops"] if tensor else peaks["hbm_gbs"]), "traffic": traffic,
            "traffic_source": f"profiles/{ncu_file} (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)" if traffic else None,
            "kernel": label, "kernel_class": dominant, "launches": d["launches"], "avg_launch_us": d["avg_us_event_bracket"],
            "algorithmic_flops_per_launch": d["flops_per_launch"], "algorithmic_bytes_per_launch": d["bytes_per_launch"],
            "peak_source": peaks["source"], "share_of_step": d["share_of_step"],
            "event_bracket_us_of_a_trivial_kernel": 1000.0 * shares["misc"]["ms"] / shares["misc"]["launches"] if "misc" in shares else None,
            "live_queries_per_iteration": {"first": hist[0], "mean": round(sum(hist) / len(hist), 2), "iterations": len(hist)},
            "timing": "CUDA events around every launch of the class on the launching stream, one extra instrumented step of the same "
                      "workload right before the timed region (bracketing every launch inside the timed region costs ~2x step time); "
                      "flops / bytes per launch follow the live queries of each iteration"}
    if "frac_in_situ" in d:
        roof["in_situ"] = {"kernel": d["kernel"], "avg_added_us": d["in_situ_us"], "frac": d["frac_in_situ"],
                           "how": "CUPTI activity records of one extra step run like the timed ones (CUDA graph + programmatic dependent "
                                  "launch): avg_added_us = end of the kernel minus end of the preceding kernel"}
    return roof, table


def dump_outputs(out_dir, outputs):
    """`--dump-outputs`: {name: (batch, n_best, width) int64 prediction or None} -> out_dir/<name>.npy as float32 (token ids are
    exact in float32).  A step that ended in one of the reference's failure modes returned no prediction and writes no file."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, pred in outputs.items():
        if pred is None:
            print(f"bench.py: the last timed step of {name} returned no prediction; {name}.npy not written", file=sys.stderr)
            continue
        np.save(d / f"{name}.npy", pred.numpy().astype(np.float32))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a B200; there is no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the one JSON line: NCCL logs to stdout (its version banner at VERSION and at WARN level)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ.pop("NCCL_DEBUG", None)
        dist.init_process_group("nccl", device_id=dev)
    wl = Workload(args.workload, args.weights, args)

    def fly_for(w):
        if args.in_flight > 0:
            return args.in_flight
        if w.kind != "greedy":
            return 12          # beam searches: 6 / 8 / 12 / 16 in flight -> 757 / 783 / 812 / 814 (beam), 881 / 931 / 954 / 938 (retro) SMILES/s
        return 3 if w.weights == "random" else 8

    n_fly = fly_for(wl)
    if args.scaling == "strong":
        n_batches = max(1, args.queries // wl.bs)
    else:
        n_batches = world * args.steps
    m = measure_workload(wl, args, local_rank, world, rank, n_fly, args.steps, args.warmup, n_batches, full=True)
    outputs = {f"{wl.key}_{wl.weights}": m["last"]}
    peaks = measured_peaks()

    line = None
    if rank == 0:
        roof, table = roofline_tables(wl, args, m, peaks) if wl.kind == "greedy" else (None, None)
        steps_equiv = n_batches / world
        line = {"metric": wl.w["metric"], "value": m["value"], "unit": "SMILES/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": m["ms"] / steps_equiv, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic",
                "config": {"workload": wl.describe(), "global_batch": world * wl.bs, "batches_timed": n_batches,
                           "parallelism": (f"dp{world}: the {n_batches} batches of the job are drawn from one queue shared by all ranks and "
                                           f"in-flight engines (no static shards); predictions all-gathered once over NCCL") if world > 1 else "single GPU",
                           "batches_in_flight": n_fly, "l2": "256 MiB buffer written before every step (L2 flush)"},
                "e2e": {"value": m["e2e_value"], "unit": "SMILES/s", "ms_per_step": m["e2e_ms"] / steps_equiv,
                        "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"]},
                "gpu_launches": m["launches"], "clocks": m["clocks"], "roofline": roof, "roofline_all": table, "kernel_shares": m["shares"],
                "decoder_calls": m["calls"], "accepted_tokens_per_call": m["accepted"] / max(m["calls"], 1),
                "produced_tokens": m["produced"], "failed_batches": m["failed_batches"], "reference_failures": m["errors"]}
        if m["one_value"] is not None:
            line["one_batch_in_flight"] = {"value": m["one_value"], "unit": "SMILES/s", "ms_per_step": m["one_ms"] / m["one_batches"],
                                           "what": "batches strictly one after the other on one engine (the kernel-level figures of `roofline` / "
                                                   "`kernels_in_situ` are measured in this mode)"}
        if m["insitu"]:
            line["kernels_in_situ"] = m["insitu"]
        parity = m["parity"]
        if world == 1 and not args.no_cpu_baseline and m["_out0"] is not None:
            nq = min(wl.bs, args.cpu_queries)
            out_sub = m["_out0"][:nq]
            if wl.kind == "beam":   # the search couples the queries of a batch (width bookkeeping): decode the sub-batch on the GPU too
                from translation_transformer_b200.model import B200Transformer
                e_ = B200Transformer(wl.cfg, wl.sd, precision=args.precision, device=local_rank)
                out_sub = wl.generator(e_).generate(wl.batch(0)[:nq].to(dev))
                e_.close()
            parity["live"], line["cpu_baseline"] = compare_with_live_reference(wl, out_sub, nq)
        checks = [p for p in parity.values() if p and p.get("checked")]
        line["parity"] = parity
        line["parity_checked"] = bool(checks)
        line["parity_ok"] = bool(checks) and all(p["top1_identical"] == p["queries"] for p in checks)

    # ---- side figures on one GPU: random-init worst case (round-1 headline) and the beam workloads ------------------------
    if world == 1 and not args.no_extra_workloads and args.scaling == "weak":
        extra = {}
        todo = []
        if args.workload == "greedy":
            other = "copy" if args.weights == "random" else "random"
            todo.append(("trained_like" if other == "copy" else "random_init_worst_case", Workload("greedy", other, args), True))
        if args.workload == "greedy":
            todo += [("beam", Workload("beam", "copy", args), False), ("retro", Workload("retro", "copy", args), False)]
        k2 = args.steps
        for key, w2, full in todo:
            try:
                n_fly2 = fly_for(w2)
                m2 = measure_workload(w2, args, local_rank, 1, 0, n_fly2, k2, args.warmup, k2, full=full)
                outputs[f"{w2.key}_{w2.weights}"] = m2["last"]
                blk = {"workload": w2.describe(), "metric": w2.w["metric"], "value": m2["value"], "unit": "SMILES/s", "steps": k2,
                       "ms_per_step": m2["ms"] / k2, "batches_in_flight": n_fly2,
                       "e2e": {"value": m2["e2e_value"], "unit": "SMILES/s", "h2d_bytes_per_step": m2["h2d"], "d2h_bytes_per_step": m2["d2h"]},
                       "one_batch_in_flight": {"value": m2["one_value"], "ms_per_step": m2["one_ms"] / m2["one_batches"]} if m2["one_value"] else None,
                       "decoder_calls_per_batch": m2["calls"] / k2, "accepted_tokens_per_call": m2["accepted"] / max(m2["calls"], 1),
                       "gpu_launches": m2["launches"], "failed_batches": m2["failed_batches"], "parity": m2["parity"]}
                if full:
                    blk["roofline"], blk["roofline_all"] = roofline_tables(w2, args, m2, peaks)
                if key == "trained_like" and not args.no_cpu_baseline and m2["_out0"] is not None:
                    nq2 = min(w2.bs, max(4, args.cpu_queries))     # real token sequences: a few more queries cost a second
                    blk["parity"]["live"], blk["cpu_baseline"] = compare_with_live_reference(w2, m2["_out0"][:nq2], nq2)
                extra[key] = blk
            except (RuntimeError, AssertionError) as ex:
                extra[key] = {"error": str(ex)[:160]}
        if line is not None:
            for key in ("trained_like", "random_init_worst_case"):
                if key in extra:
                    line[key] = extra.pop(key)
            if extra:
                line["workloads"] = extra
            for blk in [line.get("random_init_worst_case"), line.get("trained_like")] + list(line.get("workloads", {}).values()):
                for g in ((blk or {}).get("parity") or {}).values():
                    if g and g.get("checked") and g["top1_identical"] != g["queries"]:
                        line["parity_ok"] = False
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
