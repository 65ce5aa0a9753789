"""Per-call latency of the early-exit forward at small batches: eager entry points vs forward plans (CUDA graphs).

    python profiles/latency.py --out DIR [--batches 1,4,16,256] [--calls-b1 2000]

Headline configuration of bench.py (LayoutLMv3-base, concat exit + gates after all 12 layers, entropy policy with
calibrated temperatures, the entropy equivalent of 0.7 confidence), built through bench.py's own helpers.  For every
batch size B four paths, each call timed on the host clock and ended by a device synchronise:

  eager_host     model.infer on host tensors (what the reference's eval loop does, one document per call)
  plan_host      plan.infer on host tensors
  eager_device   model.infer_device on resident CUDA tensors
  plan_device    plan.infer_device on resident CUDA tensors

Calls cycle through a seeded pool of distinct documents; the paths alternate in rounds so drift on a shared machine
spreads over all of them.  Also written: the eager stage split (set_profiling, a separate pass), the card's name,
power limit and max SM clock read in the same run, and whether plan and eager results are identical on every pooled
batch.  Writes DIR/latency.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "multi-modal-early-exit_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from mmee import synth  # noqa: E402
from mmee.calibration import thresholds_for  # noqa: E402

PATHS = ("eager_host", "plan_host", "eager_device", "plan_device")
ROUNDS = 4


def card():
    o = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [x.strip() for x in o.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def calls_for(b, calls_b1):
    return {1: calls_b1, 4: max(calls_b1 // 2, 40), 16: max(calls_b1 // 5, 40)}.get(b, 40)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", default="1,4,16,256")
    ap.add_argument("--calls-b1", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("latency.py measures the GPU: no CUDA device")
    from mmee.model import B200EEForSequenceClassification

    batches = [int(x) for x in args.batches.split(",")]
    dims, ee, _, text, dtype = bench.workload("headline")
    sd = synth.make_state_dict(dims, ee, seed=0)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=max(batches), dtype=dtype)
    kind = ee.inference_strategy
    dev = torch.device("cuda", 0)
    temps = bench.calibrate_temperatures(model, dims, kind, dev)
    thr = thresholds_for(kind, bench.CONF_THRESHOLD, dims.n_labels)
    kw = dict(exit_threshold=thr, temperatures=temps)
    exit_layer = np.asarray(model.exit_layers + [dims.layers], dtype=np.float64)   # concat exit = layer 0
    result = {"workload": text, "threshold": thr, "card": card(), "rounds": ROUNDS, "batches": {}}
    print(json.dumps(result["card"]), flush=True)

    for b in batches:
        n_pool = max(8 * b, 64) if b < 256 else 2 * b
        pool = synth.make_docs(dims, n_pool, seed=2024 + b, pad=False)
        host = [{k: v[i:i + b].contiguous() for k, v in pool.items()} for i in range(0, n_pool, b)]
        resident = [{k: v.to(dev) for k, v in h.items()} for h in host]
        plan = model.plan(b)
        run = {
            "eager_host": lambda i: model.infer(**host[i], **kw),
            "plan_host": lambda i: plan.infer(**host[i], **kw),
            "eager_device": lambda i: model.infer_device(**resident[i], **kw),
            "plan_device": lambda i: plan.infer_device(**resident[i], **kw),
        }
        # plan == eager on every pooled batch, host and device forms
        identical = True
        exits = []
        for i in range(len(host)):
            e, p = model.infer(**host[i], **kw), plan.infer(**host[i], **kw)
            ed, pd = model.infer_device(**resident[i], **kw), plan.infer_device(**resident[i], **kw)
            torch.cuda.synchronize()
            identical &= bool(np.array_equal(e.exits_store, p.exits_store) and torch.equal(e.logits, p.logits)
                              and np.array_equal(e.criteria, p.criteria) and np.array_equal(e.exit_hist, p.exit_hist))
            identical &= all(torch.equal(ed[k], pd[k]) for k in ed)
            exits.append(e.exits_store)
        exits = np.concatenate(exits)
        n_calls = calls_for(b, args.calls_b1)
        per_round = max(n_calls // ROUNDS, 1)
        times = {p: [] for p in PATHS}
        for p in PATHS:
            for i in range(args.warmup):
                run[p](i % len(host))
        torch.cuda.synchronize()
        k = 0
        for _ in range(ROUNDS):
            for p in PATHS:
                for _ in range(per_round):
                    i = k % len(host)
                    k += 1
                    t0 = time.perf_counter()
                    run[p](i)
                    torch.cuda.synchronize()
                    times[p].append((time.perf_counter() - t0) * 1e3)
        model.sync()
        # stage split of the eager forward, in a pass of its own (the events perturb the timing)
        model.set_profiling(True)
        for i in range(min(per_round, 200)):
            model.infer(**host[i % len(host)], **kw)
        stages = model.last_stage_ms()
        model.set_profiling(False)
        entry = {"calls_per_path": per_round * ROUNDS, "pool_docs": n_pool, "plan_equals_eager": identical,
                 "mean_exit_layer": float(exit_layer[exits].mean()),
                 "exit_hist": np.bincount(exits, minlength=model.n_exits + 1).tolist(),
                 "eager_stage_ms": stages, "paths": {}}
        for p in PATHS:
            t = np.asarray(times[p])
            entry["paths"][p] = {"p50_ms": float(np.percentile(t, 50)), "p90_ms": float(np.percentile(t, 90)),
                                 "p99_ms": float(np.percentile(t, 99)), "mean_ms": float(t.mean()),
                                 "docs_per_s": float(b / (t.mean() / 1e3))}
        result["batches"][str(b)] = entry
        print(json.dumps({"B": b, **{p: entry["paths"][p]["p50_ms"] for p in PATHS},
                          "identical": identical, "mean_exit_layer": entry["mean_exit_layer"]}), flush=True)
        plan.close()
        del resident
        torch.cuda.empty_cache()
    result["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "latency.json"), "w") as f:
        json.dump(result, f, indent=1)
    if not all(v["plan_equals_eager"] for v in result["batches"].values()):
        raise SystemExit("plan and eager results differ")


if __name__ == "__main__":
    main()
