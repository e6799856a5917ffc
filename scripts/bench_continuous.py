"""Continuous batching vs. one batch at a time vs. engines in flight, on the greedy, beam or retro workload of bench.py.

Weights and batches are exactly the ones `bench.py --workload greedy` times (bench.Workload): product-prediction model,
vocab 288, seed 1234, batches synthetic_sources(32, 288, seed=100003 + j), bs 32, draft_len 10, n_drafts 23,
max_len 200, bf16.  Legs, all on the same batches in one process:
  (a) sequential            one engine, generate() per batch
  (b) continuous            one engine, generate_batches() for every value of --slots
  (c) in flight             k engines (InFlightDecoder), generate() per batch
  (d) continuous in flight  k engines, generate_batches() over a contiguous share of the batches each, best slots of (b)
Every leg's outputs must equal leg (a) tensor for tensor before any timing is reported.  Rates are SMILES/s from the host
clock around work that ends in a device synchronise; every shape is warmed up first (graphs are captured lazily).

    python scripts/bench_continuous.py --weights copy --batches 24 --out profiles/continuous_copy.json

--workload beam / retro runs the speculative beam searches of bench.py (configs[2]: bs 4, n_best 5; configs[3]: 6+6 layers,
bs 8, n_best 10) with the same legs; their slot sweep and engine counts default to multiples of the batch size and to the
12 engines bench.py keeps in flight for them, leg (d) is skipped unless --cont-inflight is given.  Every leg also records the
device memory its engines hold after the run, and leg (b) the mean and maximum query slots in use per iteration; leg (a)
of a beam search reports the bs slots it holds as `slots_held` (its generate() keeps no per-iteration history).

    python scripts/bench_continuous.py --workload retro --weights copy --batches 48 --out profiles/r4_continuous_beam_retro.json

--workload std_beam / std_retro run the standard beam search (TranslationInferenceBeamSearch, beam_size = n_best) on the
model, weights and batches of the beam / retro workloads, with the legs and defaults of those workloads.

    python scripts/bench_continuous.py --workload std_beam --weights copy --batches 48 --out profiles/r5_continuous_std_beam_copy.json

--workload std_greedy runs the standard greedy decoding (TranslationInferenceGreedy) on the model, weights and batches of
the greedy workload, with the greedy workload's engines in flight and a slot sweep of 1, 2, 4, 8 and 16 x bs (no leg (d)
unless --cont-inflight is given).

    python scripts/bench_continuous.py --workload std_greedy --weights copy --batches 24 --out profiles/r6_continuous_std_greedy_copy.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

import bench  # noqa: E402
from translation_transformer_b200.decoding import TranslationInferenceBeamSearch, TranslationInferenceGreedy  # noqa: E402
from translation_transformer_b200.model import B200Transformer  # noqa: E402
from translation_transformer_b200.pipeline import InFlightDecoder  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, max_sm, sm = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"card": name, "power_limit": power, "sm_clock_max": max_sm, "sm_clock_at_start": sm}


def history(eng):
    buf = (C.c_int32 * 200000)()
    n = eng.lib.ttb_engine_get_history(eng._h, buf, len(buf))
    return list(buf[:n])


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return res, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="greedy", choices=["greedy", "beam", "retro", "std_greedy", "std_beam", "std_retro"])
    ap.add_argument("--weights", default="copy", choices=["copy", "random"])
    ap.add_argument("--batches", type=int, default=24)
    ap.add_argument("--slots", default=None, help="comma-separated slot counts (default greedy: 32,48,64,96,128; std_greedy and beam searches: 1,2,4,8,16 x bs)")
    ap.add_argument("--inflight", default=None, help="engines in flight (default greedy and std_greedy: 3,8; beam searches: 12)")
    ap.add_argument("--cont-inflight", default=None, help="continuous loops in flight (default greedy: 2,4; std_greedy and beam searches: none)")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    std = a.workload.startswith("std_")
    base = a.workload[len("std_"):] if std else a.workload
    greedy = base == "greedy"
    argv, sys.argv = sys.argv, ["bench.py", "--workload", base, "--weights", a.weights]
    bargs = bench.parse()
    sys.argv = argv
    wl = bench.Workload(base, a.weights, bargs)
    if std and greedy:   # the standard greedy decoding on the workload's model and batches
        wl.generator = lambda eng: TranslationInferenceGreedy(eng, bargs.max_len, bench.PAD, bench.BOS, bench.EOS)
    elif std:   # the standard beam search on the workload's model and batches
        wl.generator = lambda eng: TranslationInferenceBeamSearch(eng, wl.n_best, bargs.max_len, bench.PAD, bench.BOS, bench.EOS)
    if a.slots is None:
        a.slots = "32,48,64,96,128" if a.workload == "greedy" else ",".join(str(k * wl.bs) for k in (1, 2, 4, 8, 16))
    if a.inflight is None:
        a.inflight = "3,8" if greedy else "12"
    if a.cont_inflight is None:
        a.cont_inflight = "2,4" if a.workload == "greedy" else ""
    dev = torch.device("cuda", 0)
    batches = [wl.batch(j).to(dev) for j in range(a.batches)]
    n_smiles = sum(b.shape[0] for b in batches)
    std_name = "standard greedy decoding, on: " if greedy else "standard beam search, beam_size = n_best, on: "
    res = {"workload": (std_name if std else "") + wl.describe(), "batches": a.batches, "bs": wl.bs, "weights": a.weights, **gpu_info()}
    if not greedy:
        res["n_best"] = wl.n_best

    def engine():
        return B200Transformer(wl.cfg, wl.sd, precision="bf16", device=0)

    def mem_of(make):   # device memory an engine holds after a warm run
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        eng = make()
        return eng, free0

    # (a) sequential
    eng0, free0 = mem_of(engine)
    gen0 = wl.generator(eng0)
    for b in batches[:2]:
        gen0.generate(b)
    ref, t = timed(lambda: [gen0.generate(b) for b in batches])
    h = []
    for b in batches[:4]:
        gen0.generate(b)
        h += history(eng0)
    torch.cuda.synchronize()
    res["a_sequential"] = {"smiles_per_s": n_smiles / t, "s": t}
    if greedy:
        res["a_sequential"].update(mean_live=sum(h) / len(h), max_live=max(h))
    else:   # generate() of the beam search keeps no per-iteration history: it holds its bs query slots throughout
        res["a_sequential"]["slots_held"] = wl.bs
    res["a_sequential"]["engine_bytes"] = free0 - torch.cuda.mem_get_info(0)[0]

    # (b) continuous, one engine per slots value (memory per engine then includes that slots value's workspace)
    res["b_continuous"] = []
    best = None
    for slots in [int(x) for x in a.slots.split(",")]:
        eng, free0 = mem_of(engine)
        gen = wl.generator(eng)
        gen.generate_batches(batches[:6], slots=slots)        # warm-up: graphs of every bucket this slots value uses
        out, t = timed(lambda: gen.generate_batches(batches, slots=slots))
        assert all(torch.equal(x, y) for x, y in zip(ref, out)), f"continuous slots={slots} differs from generate()"
        h = history(eng)
        r = {"slots": slots, "smiles_per_s": n_smiles / t, "s": t, "mean_live": sum(h) / len(h), "max_live": max(h),
             "iterations": len(h), "engine_bytes": free0 - torch.cuda.mem_get_info(0)[0]}
        res["b_continuous"].append(r)
        if best is None or r["smiles_per_s"] > best["smiles_per_s"]:
            best = r
        eng.close()
        del eng, gen
        torch.cuda.empty_cache()
        print(json.dumps(r), flush=True)

    # (c) engines in flight
    res["c_in_flight"] = []
    for k in [int(x) for x in a.inflight.split(",") if x]:
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        engs = [engine() for _ in range(k)]
        dec = InFlightDecoder([wl.generator(e) for e in engs], device=dev)
        list(dec.map(batches[:2 * k]))
        out, t = timed(lambda: list(dec.map(batches)))
        assert all(torch.equal(x, y) for x, y in zip(ref, out)), f"in-flight k={k} differs from generate()"
        torch.cuda.synchronize()
        r = {"engines": k, "smiles_per_s": n_smiles / t, "s": t}
        if not greedy:
            r["engine_bytes"] = free0 - torch.cuda.mem_get_info(0)[0]
        res["c_in_flight"].append(r)
        dec.close()
        for e in engs:
            e.close()
        torch.cuda.empty_cache()

    # (d) continuous loops in flight: each engine decodes a contiguous share of the batches on its own stream
    res["d_continuous_in_flight"] = []
    for k in [int(x) for x in a.cont_inflight.split(",") if x]:
        engs = [engine() for _ in range(k)]
        gens = [wl.generator(e) for e in engs]
        streams = [torch.cuda.Stream(device=dev) for _ in range(k)]
        share = (len(batches) + k - 1) // k
        parts = [batches[i * share:(i + 1) * share] for i in range(k)]

        def run(i, outs):
            torch.cuda.set_device(dev)
            with torch.cuda.stream(streams[i]):
                outs[i] = gens[i].generate_batches(parts[i], slots=best["slots"]) if parts[i] else []
                streams[i].synchronize()

        def all_parts():
            outs = [None] * k
            th = [threading.Thread(target=run, args=(i, outs)) for i in range(k)]
            for x in th:
                x.start()
            for x in th:
                x.join()
            return [o for part in outs for o in part]

        all_parts()
        out, t = timed(all_parts)
        assert all(torch.equal(x, y) for x, y in zip(ref, out)), f"continuous in flight k={k} differs from generate()"
        res["d_continuous_in_flight"].append({"engines": k, "slots": best["slots"], "smiles_per_s": n_smiles / t, "s": t})
        for e in engs:
            e.close()
        torch.cuda.empty_cache()

    res["best_slots"] = best["slots"]
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
