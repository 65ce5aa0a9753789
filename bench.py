#!/usr/bin/env python
"""Benchmark of the early-exit inference hot path (BASELINE.json metric: documents/sec at a fixed
calibrated exit threshold; exit-layer agreement %).

    python bench.py --gpus N --steps K --warmup W                     # headline: BASELINE.json configs[1]
    python bench.py --config sweep|large|image_only|fp32 ...          # the other BASELINE configs / the fp32 mode
    python bench.py --impl reference --gpus N --steps K ...           # the reference's CPU implementation (oracle port)
    python bench.py ... --dump-outputs DIR                             # also write the last timed step's results as .npy

A step = one pass of the hot path over one batch of synthetic RVL-CDIP-shaped documents
(512 text tokens + boxes + 224x224 image, 16 classes).  Workloads (BASELINE.json `configs`):

  headline    configs[1]: LayoutLMv3-base, learned exit gates after every layer (+ the text_visual_concat embedding
              exit), batch 256 per GPU, bf16 tensor-core math, entropy-threshold policy with per-exit temperature
              calibration.  Weak scaling (256 documents per GPU at every N).
  sweep       configs[2]: LayoutLMv3-base, ramps, max-confidence policy, 8192 documents sharded data-parallel over the
              N GPUs (strong scaling: 8192 / N per GPU, micro-batches of <= 1024), calibrated thresholds 0.5 ... 0.99:
              per threshold docs/s, mean exit layer, algorithmic TFLOP/s of the layers the documents really ran.
  large       configs[3]: LayoutLMv3-large (24 layers, hidden 1024), ramps every 2 layers, 512 documents per GPU
              (4096 on 8 GPUs).
  image_only  configs[4]: patch tokens only (197 tokens per document), ramps after every layer, 2048 documents per GPU
              (16384 on 8 GPUs).
  fp32        the headline workload in the fp32-parity engine mode (split-bf16 operands, logits within 1e-4).

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "multi-modal-early-exit_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mmee import synth  # noqa: E402
from mmee.calibration import spread_temperatures, thresholds_for  # noqa: E402
from mmee.config import ExitConfig, ModelDims  # noqa: E402

METRIC = "docs/sec @ calibrated exit threshold"
CONF_THRESHOLD = 0.7          # calibrated-confidence level the exit threshold is derived from
SWEEP_THRESHOLDS = (0.5, 0.6, 0.7, 0.8, 0.9, 0.95, 0.99)
SWEEP_DOCS = 8192
AGREEMENT_DOCS = 16           # documents of the timed batch re-run through the oracle (exit_agreement)
CPU_SAMPLE_DOCS = 16          # SURVEY.md §8(d): config 1 exactly (B = 16), 1 warm-up + 3 timed, median
DUMP_LIMIT_BYTES = 64 << 20   # --dump-outputs: total size of the arrays written


def workload(config: str):
    """-> (dims, ee, batch_per_gpu, text, dtype)"""
    if config in ("headline", "fp32"):
        dims = ModelDims.base()
        ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(1, dims.layers + 1)),
                                       encoder_layer_strategy="gate", inference_strategy="entropy"))
        text = ("LayoutLMv3-base, concat exit + learned exit gates after all 12 layers, entropy-threshold policy "
                "with temperature calibration, 512 tokens + 224x224 image, 16 classes, batch 256 per GPU")
        if config == "fp32":
            text += " — fp32-parity engine mode (split-bf16 operands on the tensor cores)"
        return dims, ee, 256, text, ("fp32" if config == "fp32" else "bf16")
    if config == "sweep":
        dims = ModelDims.base()
        ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(1, dims.layers + 1)),
                                       encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
        return dims, ee, 1024, ("LayoutLMv3-base, concat exit + ramps after all 12 layers, max-confidence policy with "
                                "temperature calibration, 8192 documents sharded over the GPUs, threshold sweep "
                                "0.5-0.99, 512 tokens + 224x224 image, 16 classes"), "bf16"
    if config == "large":
        dims = ModelDims.large()
        ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(2, dims.layers + 1, 2)),
                                       encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
        return dims, ee, 512, ("LayoutLMv3-large (24 layers, hidden 1024), concat exit + ramps every 2 layers, "
                               "max-confidence policy with temperature calibration, 512 tokens + 224x224 image, "
                               "16 classes, batch 512 per GPU (4096 on 8 GPUs)"), "bf16"
    if config == "image_only":
        dims = ModelDims.base(n_text=0)
        ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(1, dims.layers + 1)),
                                       encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
        return dims, ee, 2048, ("image-only path (IC_only.py-style: 196 patch tokens + CLS, no text), LayoutLMv3-base "
                                "encoder, concat exit + ramps after all 12 layers, max-confidence policy with "
                                "temperature calibration, 224x224 image, 16 classes, batch 2048 per GPU (16384 on 8 GPUs)"), "bf16"
    raise ValueError(config)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            j = json.load(f)
        return dict(hbm=j.get("hbm_gbs", 6650.0), tf_burst=j.get("bf16_tflops", 1590.0),
                    tf_sust=j.get("bf16_tflops_sustained", 1400.0), source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback")


class ClockSampler:
    """Samples the SM clock + throttle reasons of one GPU while the timed region runs: in-process NVML (cheap enough
    for a 20 ms period, no driver-lock storms when 8 ranks share a box), `nvidia-smi` as the fallback."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index: int, enabled: bool = True):
        self.index = index
        self.enabled = enabled
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.source = None
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _nvml_handle(self):
        import pynvml

        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _run(self):
        try:
            nv, h = self._nvml_handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.source = "nvml"
            while not self._stop.is_set():
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(nm)
                self._stop.wait(0.02)
            return
        except Exception:
            pass
        self.source = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(o[0]))
                self.max_mhz = float(o[1])
                for nm, v in zip(names, o[2:]):
                    if v.strip().lower() == "active":
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        if self.enabled:
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.enabled:
            self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "source": self.source}


def layer_flops(dims: ModelDims):
    """SURVEY.md §8(d): algorithmic FLOPs per document-layer (2 M N K per GEMM) and of the patch embedding."""
    S, H, I = dims.seq, dims.hidden, dims.inter
    return dict(linear=2.0 * S * (4 * H * H + 2 * H * I), attn=4.0 * S * S * H,
                patch=2.0 * dims.n_patch * (dims.channels * dims.patch ** 2) * H)


def reached_per_layer(hist, exit_layers, n_layers, n_docs):
    """documents entering encoder layer l (1-based) given the exit histogram (index = exit number)."""
    out = []
    for l in range(1, n_layers + 1):
        left_before = sum(int(hist[i]) for i, el in enumerate(exit_layers) if el < l)
        out.append(n_docs - left_before)
    return out


def unpack_results(rows, K: int):
    """Packed result rows [..., K + 2] (`mmee.dist.pack_results`) -> logits, exit index, criterion."""
    return {"logits": rows[..., :K], "exit_index": rows[..., K].astype(np.int64), "criterion": rows[..., K + 1]}


def dump_outputs(out_dir: str, arrays) -> None:
    """`--dump-outputs`: write the results the timed path returned in its last step as `<out_dir>/<name>.npy` (floats
    as they are, integer arrays as float64), so that two builds can be compared output for output on the same seeded
    inputs.  The temperatures and thresholds come from the build's own calibration pass; they are written too, so
    that a difference in exit indices can be told apart from a difference in calibration."""
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        out[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_port_time(dims, ee, sd, docs, threads: int) -> float:
    """One dense forward of the oracle port (reference algorithm, torch CPU fp32, every exit for every document)."""
    from oracle import port

    torch.set_num_threads(threads)
    with torch.no_grad():
        t0 = time.perf_counter()
        port.forward(sd, dims, ee, docs)
        return time.perf_counter() - t0


def cpu_baseline_config1(threads: int):
    """SURVEY.md §8(d) recipe: BASELINE configs[0] exactly — LayoutLMv3-base, ramps after every layer (13 exits + the
    final classifier), B = 16 padded documents, fp32, all host threads; 1 warm-up + 3 timed forwards, median."""
    dims = ModelDims.base()
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(1, dims.layers + 1)),
                                   encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
    sd = synth.make_state_dict(dims, ee, seed=0)
    docs = synth.make_docs(dims, CPU_SAMPLE_DOCS, seed=1, pad=True)
    cpu_port_time(dims, ee, sd, {k: v[:2] for k, v in docs.items()}, threads)          # warm-up (2 documents)
    times = [cpu_port_time(dims, ee, sd, docs, threads) for _ in range(3)]
    med = statistics.median(times)
    return {"value": CPU_SAMPLE_DOCS / med, "unit": "docs/s", "cores": threads, "kind": "port",
            "torch_threads": torch.get_num_threads(), "os_cpu_count": os.cpu_count(),
            "sample": (f"BASELINE configs[0]: {CPU_SAMPLE_DOCS} padded documents, base model with 13 ramps, dense forward "
                       f"(the reference never skips work), torch CPU fp32; 1 warm-up + 3 timed, median {med:.2f} s "
                       f"(runs {', '.join(f'{t:.2f}' for t in times)} s)")}


def run_reference(args):
    """`--impl reference`: the reference's own CPU path for the same workload.  /root/reference (pure Python on
    HF transformers) does not exist on the GPU box, so this times oracle/port.py — validated bit-exact against
    the unmodified reference by tests/test_oracle.py — with all host threads, on a bounded sample per step
    (16 documents, the batch of BASELINE configs[0])."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dims, ee, _, text, _ = workload(args.config)
    sd = synth.make_state_dict(dims, ee, seed=0)
    threads = os.cpu_count() or 1
    n_docs = CPU_SAMPLE_DOCS if args.config != "large" else 4
    docs = synth.make_docs(dims, n_docs, seed=1, pad=False)
    for _ in range(max(min(args.warmup, 1), 0)):                     # one warm-up forward is enough on the CPU
        cpu_port_time(dims, ee, sd, {k: v[:2] for k, v in docs.items()}, threads)
    times = [cpu_port_time(dims, ee, sd, docs, threads) for _ in range(args.steps)]
    ms = 1000.0 * sum(times) / len(times)
    v = n_docs / (ms / 1000.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "docs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": text, "bench_config": args.config,
                   "sample": f"{n_docs} documents per step, all exits computed (the reference never skips work)"},
        "cpu_baseline": {"value": v, "unit": "docs/s", "cores": threads, "kind": "port",
                         "sample": f"{n_docs} docs/step x {args.steps} steps, torch CPU fp32, median step "
                                   f"{statistics.median(times):.2f} s"},
        "e2e": {"value": v, "unit": "docs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def agreement_vs_oracle(model, dims, ee, sd, docs, exits_timed, temps, thr, kind):
    """`exit_agreement`: the first AGREEMENT_DOCS documents of the timed batch through the oracle (port + policy port)
    with the bench's own temperatures and threshold.  Agreement over all of them, and over the decisive ones: at every
    exit the oracle's criterion keeps more than 1.5x the engine's own criterion error (measured on its dense logits
    for the same documents) from the threshold."""
    from oracle import policy_port, port

    n = min(AGREEMENT_DOCS, docs["pixel_values"].shape[0])
    sub = {k: v[:n] for k, v in docs.items()}
    dev = torch.device("cuda", model.device_index)
    dense = model.infer(**{k: v.to(dev) for k, v in sub.items()}, exit_threshold=thr, temperatures=temps,
                        early_exit=False, return_all=True)
    eng = dense.all_exit_logits.cpu().numpy().astype(np.float64)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        ref = port.forward(sd, dims, ee, sub)["exit_logits"].numpy().astype(np.float64)
    ref_cal = policy_port.temperature_scale(ref, temps)
    eng_cal = policy_port.temperature_scale(eng, temps)
    want, _, crit_ref = policy_port.exit_policy_vectorised(ref_cal, thr, kind)
    crit_eng = policy_port.criterion(eng_cal, kind)
    err = np.abs(crit_eng - crit_ref)[:-1]
    margin = np.abs(crit_ref[:-1] - thr)
    decisive = (margin > 1.5 * err + 1e-7).all(axis=0)
    got = np.asarray(exits_timed[:n])
    agree = got == want
    layers = np.array(model.exit_layers + [dims.layers])
    return {"n_docs": int(n), "all_docs": float(agree.mean()),
            "decisive": float(agree[decisive].mean()) if decisive.any() else None,
            "decisive_frac": float(decisive.mean()),
            "margin": "at every exit |oracle criterion - threshold| > 1.5 x |engine criterion - oracle criterion| "
                      "(engine dense logits of the same documents)",
            "max_logit_err": float(np.abs(eng - ref).max()),
            "predicted_class_agreement": float((eng.argmax(-1) == ref.argmax(-1)).mean()),
            "exit_layers_engine": np.clip(layers[got], 0, None).tolist(),
            "exit_layers_oracle": np.clip(layers[want], 0, None).tolist(),
            "oracle": "oracle/port.py + oracle/policy_port.py (pinned to the reference goldens)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mmee", choices=["mmee", "reference"])
    ap.add_argument("--config", default="headline", choices=["headline", "sweep", "large", "image_only", "fp32"])
    ap.add_argument("--batch", type=int, default=0, help="documents per GPU per step (default: the config's)")
    ap.add_argument("--threshold", type=float, default=CONF_THRESHOLD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-agreement", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step, gathered over the GPUs, and the calibrated "
                         "temperatures and thresholds to DIR/<name>.npy (written by rank 0; the mmee path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "mmee":
        ap.error("--dump-outputs writes the results of the mmee path only")
    args.warmup = max(args.warmup, 3) if args.impl == "mmee" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        warm = torch.zeros(8, device=dev)                # NCCL communicator set-up (seconds) happens here, not in a timed
        dist.all_reduce(warm)                            # or clock-sampled region
        dist.all_gather_into_tensor(torch.empty(8 * world, device=dev), warm)
        torch.cuda.synchronize()

    if args.config == "sweep":
        run_sweep(args, world, rank, local, dev)
    else:
        run_single(args, world, rank, local, dev)
    if world > 1:
        dist.destroy_process_group()


def calibrate_temperatures(model, dims, kind, dev, n_docs=64):
    """Calibration pass (dense) on a held-out synthetic batch: per-exit temperatures such that the median calibrated
    criterion rises with depth (SURVEY.md §8(d)); the same on every rank (same seed)."""
    cal_docs = synth.make_docs(dims, min(model.max_batch, n_docs), seed=12345, pad=False)
    cal = model.infer(**{k: v.to(dev) for k, v in cal_docs.items()}, exit_threshold=-1.0 if kind == "entropy" else 2.0,
                      early_exit=False, return_all=True)
    return spread_temperatures(cal.all_exit_logits.cpu().numpy(), kind)


def timed_region(fn, steps, warmup, world, dev, finish=None, before_timed=None):
    """W untimed + K timed calls of fn bracketed by barrier + synchronize on both sides, CUDA events on the current
    stream, MAX over ranks.  `finish` (optional) runs inside the timed region after the last step (final gather);
    `before_timed` (optional) runs after the warm-up, outside the timed region."""
    import torch.distributed as dist

    for _ in range(warmup):
        fn()
    if finish:
        finish()
    torch.cuda.synchronize()
    if before_timed:
        before_timed()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for _ in range(steps):
        last = fn()
    if finish:
        last = finish() or last
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps, last


def run_single(args, world, rank, local, dev):
    """headline / large / image_only / fp32: one batch per GPU per step (weak scaling)."""
    import torch.distributed as dist

    from mmee.model import B200EEForSequenceClassification

    dims, ee, B, text, dtype = workload(args.config)
    if args.batch:
        B = args.batch
    sd = synth.make_state_dict(dims, ee, seed=0)
    model = B200EEForSequenceClassification(dims, ee, sd, device=local, max_batch=B, dtype=dtype)
    kind = ee.inference_strategy
    E1 = model.n_exits + 1
    K = dims.n_labels
    temps = calibrate_temperatures(model, dims, kind, dev)
    thr = thresholds_for(kind, args.threshold, K)

    docs = synth.make_docs(dims, B, seed=1 + 1000 * rank, pad=False)
    dev_docs = {k: v.to(dev) for k, v in docs.items()}
    pin_docs = {k: v.pin_memory() for k, v in docs.items()}
    steps = args.steps

    # ---- device-resident timing.  N > 1: the job's results (logits | exit index | criterion per document) are gathered
    # over NVLink on NCCL's stream after every step WITHOUT a host round-trip; the ranks therefore do not run in
    # lock-step (a slower board only delays the gather it takes part in), and the whole job's results are read back to
    # the host once, at the end of the timed region ("final gather").
    from mmee.dist import JobGatherer, pack_results

    # One job = `steps` batches per GPU.  Every step is enqueued without waiting (infer_device: results stay on the GPU)
    # and its packed per-document results go into a local device ring; at the end of the job the rings are all-gathered
    # (N > 1: one NCCL call) and the whole job's results are read back to the host ONCE, inside the timed region
    # ("final gather", SURVEY.md §8e).  The same code path at every N.
    cap = max(steps, args.warmup)
    jg = JobGatherer(B, K + 2, E1, cap, dev) if world > 1 else None
    ring1 = torch.empty((cap, B, K + 2), dtype=torch.float32, device=dev) if world == 1 else None
    hist1 = torch.zeros((E1,), dtype=torch.int64, device=dev)
    state = {"last": None, "i": 0}

    def step_device():
        r = model.infer_device(**dev_docs, exit_threshold=thr, temperatures=temps)
        packed = pack_results(r["logits"], r["exit_index"], r["criterion"])
        if world > 1:
            jg.push(packed, r["hist"])
        else:
            ring1[state["i"] % cap].copy_(packed)
            hist1.add_(r["hist"])
        state["i"] += 1
        state["last"] = r
        return r

    def finish_device():
        if world > 1:
            fin = jg.finish()                            # waits for the gathers; ONE read-back of every step's results
            results, job_hist = fin["results"], fin["exit_hist"].numpy()
        else:
            results, job_hist = ring1.cpu(), hist1.cpu().numpy()
            hist1.zero_()
        model.sync()                                     # folds the stage events, surfaces device-side error flags
        state["i"] = 0
        r = dict(state["last"])
        r["exit_hist"] = r["hist"].cpu().numpy()
        r["exits_store"] = r["exit_index"].cpu().numpy()
        r["job_results"] = results
        r["job_hist"] = job_hist
        return r

    with ClockSampler(local, enabled=True) as clk:
        ms_step, res = timed_region(step_device, steps, args.warmup, world, dev, finish_device,
                                    before_timed=lambda: model.set_profiling(True))
    stage = model.last_stage_ms()          # per-stage CUDA-event times, averaged over the timed steps
    launches = model.last_launch_count()
    model.set_profiling(False)
    if args.dump_outputs and rank == 0:    # the last step's rows of the job results: every rank's batch, in rank order
        out = unpack_results(res["job_results"][(steps - 1) % cap].numpy(), K)
        out["exit_hist"] = np.bincount(out["exit_index"], minlength=E1)
        dump_outputs(args.dump_outputs, dict(out, temperatures=temps, thresholds=np.atleast_1d(thr)))
    value = world * B / (ms_step / 1000.0)
    clocks_all = [clk.summary()]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, clk.summary())
        clocks_all = gathered

    # ---- data-parallel consistency on the hardware (SURVEY.md §4 item 4): every rank re-runs rank 0's shard and
    # compares it bit for bit with rank 0's rows of the gathered job results
    dp_consistency = None
    if world > 1:
        docs0 = synth.make_docs(dims, B, seed=1, pad=False)
        r0 = model.infer_device(**{k: v.to(dev) for k, v in docs0.items()}, exit_threshold=thr, temperatures=temps)
        mine = pack_results(r0["logits"], r0["exit_index"], r0["criterion"]).cpu()
        theirs = res["job_results"][(steps - 1) % res["job_results"].shape[0], :B]
        ok = torch.tensor([1 if torch.equal(mine, theirs) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        dp_consistency = {"checked": True, "bit_exact_on_all_ranks": bool(ok.item()), "ranks": world,
                          "what": "every rank re-ran rank 0's 256-document shard and compared logits, exit index and "
                                  "criterion with rank 0's rows of the NCCL-gathered job results"}

    # ---- end to end through the public API with HOST buffers
    e2e = None
    if not args.no_e2e:
        n_e2e = max(2, min(steps, 5))
        if world == 1:
            def step_host():
                return model.infer(**pin_docs, exit_threshold=thr, temperatures=temps)
            api = "B200EEForSequenceClassification.infer (blocking, host tensors in, host results out)"
        else:
            out_all = torch.empty((world * B, K + 2), dtype=torch.float32, device=dev)

            def step_host():
                up = {k: v.to(dev, non_blocking=True) for k, v in pin_docs.items()}
                r = model.infer_device(**up, exit_threshold=thr, temperatures=temps)
                dist.all_gather_into_tensor(out_all, pack_results(r["logits"], r["exit_index"], r["criterion"]))
                return out_all.cpu()                 # the job's results on the host: the step ends here
            api = ("pinned host tensors -> B200EEForSequenceClassification.infer_device -> NCCL all_gather of the "
                   "job's results -> host, every step")
        ms_block, _ = timed_region(step_host, n_e2e, 2, world, dev)
        h2d = sum(int(v.numel() * v.element_size()) for k, v in pin_docs.items() if k != "labels")
        d2h = (B * K * 4 + B * 4 + B * 4 + E1 * 8) if world == 1 else world * B * (K + 2) * 4
        e2e = {"value": world * B / (ms_block / 1000.0), "unit": "docs/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": ms_block, "api": api}
        if world == 1:
            # pipelined form: infer_submit / infer_collect with two batches in flight (upload of batch n+1 overlaps the
            # forward of batch n), wall clock including pipeline fill and drain
            pend = []

            def step_pipelined():
                pend.append(model.infer_submit(**pin_docs, exit_threshold=thr, temperatures=temps))
                if len(pend) == 2:
                    return model.infer_collect(pend.pop(0))
                return None

            def drain():
                while pend:
                    model.infer_collect(pend.pop(0))

            for _ in range(2):
                step_pipelined()
            drain()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                step_pipelined()
            drain()                                    # every submitted step has been read back when the clock stops
            torch.cuda.synchronize()
            ms_pipe = (time.perf_counter() - t0) * 1000.0 / n_e2e
            e2e.update({"pipelined_value": B / (ms_pipe / 1000.0), "pipelined_ms_per_step": ms_pipe,
                        "pipelined_api": "infer_submit/infer_collect, 2 batches in flight, wall clock incl. pipeline fill and drain"})

    # ---- SURVEY.md §8(d) primary input recipe: text lengths ~ U{64..512}, padded to 512 (the headline above is its
    # all-512 no-pad variant, the harder case: no key tile is ever skipped)
    padded = None
    if world == 1 and not args.no_e2e and dims.n_text > 0:
        pdocs = synth.make_docs(dims, B, seed=7, pad=True)
        pdev = {k: v.to(dev) for k, v in pdocs.items()}
        ms_pad, res_p = timed_region(lambda: model.infer(**pdev, exit_threshold=thr, temperatures=temps),
                                     max(2, min(steps, 4)), 2, world, dev)
        ph = np.asarray(res_p.exit_hist, dtype=np.float64)
        padded = {"value": B / (ms_pad / 1000.0), "unit": "docs/s", "ms_per_step": ms_pad,
                  "mean_real_text_tokens": float(pdocs["attention_mask"].sum(1).float().mean()),
                  "mean_exit_layer": float(np.dot(ph, np.clip(np.array(model.exit_layers + [dims.layers]), 0, None)) / ph.sum()),
                  "note": "same engine, thresholds and temperatures; ragged documents: rows of padded text tokens are dropped after the embedding stage (no GEMM / LayerNorm / attention work for them)"}

    # ---- roofline of the dominant kernel (tcgen05 GEMM): algorithmic FLOPs of the docs that reached each layer
    hist = res["exit_hist"].astype(np.int64)
    fl = layer_flops(dims)
    exit_layers = model.exit_layers
    reached = reached_per_layer(hist, exit_layers, dims.layers, B)
    gemm_flops = sum(reached) * fl["linear"] + B * fl["patch"]
    attn_flops = sum(reached) * fl["attn"]
    pk = peaks()
    gemm_tf = gemm_flops / (stage["gemm"] / 1000.0) / 1e12 if stage.get("gemm") else None
    attn_tf = attn_flops / (stage["attention"] / 1000.0) / 1e12 if stage.get("attention") else None
    traffic, traffic_src, att_traffic = None, None, None
    tj = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tj) and args.config == "headline" and B == 256:   # ncu --set full capture of the same workload
        with open(tj) as f:
            tr = json.load(f)
        traffic = tr.get("gemm_mean_dram_bytes_per_launch")
        traffic_src = (f"ncu dram__bytes_read.sum+dram__bytes_write.sum, mean of the 4 GEMM launches of one layer at "
                       f"{tr.get('docs')} docs (profiles/traffic.json, capture {tr.get('capture')})")
        att_traffic = tr.get("attention")
    mma_factor = 3.0 if dtype == "fp32" else 1.0           # fp32 mode: three bf16 tensor-core products per contraction
    roofline = {"bound": "tensor", "kernel": "gemm_tc_pair_kernel (QKV / out-proj / MLP-up+GELU / MLP-down; tcgen05 cta_group::2)",
                "achieved": gemm_tf, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                "frac": (gemm_tf / pk["tf_sust"]) if gemm_tf else None, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": pk["source"] + " (sustained: kernel timed inside a long step)",
                "attention": {"achieved": attn_tf, "unit": "TFLOP/s", "frac": (attn_tf / pk["tf_sust"]) if attn_tf else None,
                              "traffic": att_traffic},
                "stage_ms": stage, "stage_ms_note": "CUDA events between the stages of every timed step, averaged over the timed steps",
                "whole_step_frac": (gemm_flops + attn_flops) / (ms_step / 1000.0) / 1e12 / pk["tf_sust"]}
    if dtype == "fp32":
        roofline["note"] = ("algorithmic (fp32-equivalent) FLOPs; the tensor cores execute 3x that in bf16 products: "
                            f"tensor-pipe rate = {mma_factor:g} x achieved")
        roofline["tensor_pipe_tflops"] = gemm_tf * mma_factor if gemm_tf else None

    if rank == 0:
        cpu = None
        agreement = None
        if world == 1 and not args.no_agreement:
            exits_timed = res["exits_store"]
            agreement = agreement_vs_oracle(model, dims, ee, sd, docs, exits_timed, temps, thr, kind)
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_config1(os.cpu_count() or 1)
        layers_of_exit = np.clip(np.array(exit_layers + [dims.layers]), 0, None)
        mean_depth = float(np.dot(hist, layers_of_exit) / hist.sum())
        line = {
            "metric": METRIC, "value": value, "unit": "docs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": {"workload": text, "bench_config": args.config, "global_batch": world * B, "parallelism": f"dp{world}",
                       "criterion": kind, "threshold": thr, "calibrated_confidence_level": args.threshold,
                       "temperatures": [round(float(t), 5) for t in temps],
                       "exit_hist_rank0": hist.tolist(), "mean_exit_layer_rank0": mean_depth,
                       "l2_policy": "working set per layer (attention bias + activations, several GB) exceeds the 126 MB L2"},
            "clocks": clocks_all[0], "e2e": e2e, "gpu_launches": int(launches) * args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "exit_agreement": agreement, "padded_variant": padded,
        }
        if world > 1:
            line["dp_consistency"] = dp_consistency
            line["clocks_per_gpu"] = clocks_all
            line["gather"] = ("every step's [256, K+2] results are kept in a local device ring; ONE NCCL all_gather of "
                              "the rings + one all_reduce of the exit histogram + one device->host read-back at the "
                              "end of the timed region (no collective while the job computes)")
        line["config"]["job"] = (f"{args.steps} batches per GPU enqueued back to back; every step's per-document results "
                                 "are kept in a device ring and read back to the host once, inside the timed region")
        print(json.dumps(line), flush=True)


def run_sweep(args, world, rank, local, dev):
    """BASELINE configs[2]: 8192 documents sharded over the GPUs (strong scaling), thresholds 0.5 ... 0.99.  One step =
    the whole sweep (every threshold over every document of the shard)."""
    import torch.distributed as dist

    from mmee.dist import pack_results
    from mmee.model import B200EEForSequenceClassification

    dims, ee, MB, text, dtype = workload("sweep")
    n_total = SWEEP_DOCS
    n_local = n_total // world
    MB = min(args.batch or MB, n_local)
    n_mb = (n_local + MB - 1) // MB
    sd = synth.make_state_dict(dims, ee, seed=0)
    model = B200EEForSequenceClassification(dims, ee, sd, device=local, max_batch=MB, dtype=dtype)
    kind = ee.inference_strategy
    K = dims.n_labels
    E1 = model.n_exits + 1
    temps = calibrate_temperatures(model, dims, kind, dev)
    # the shard: micro-batches of distinct documents, resident in HBM (4.9 GB of pixels for all 8192)
    shards = []
    for m in range(n_mb):
        n = min(MB, n_local - m * MB)
        d = synth.make_docs(dims, n, seed=100 + rank * n_mb + m, pad=False)
        shards.append({k: v.to(dev) for k, v in d.items()})
    out_all = torch.empty((world * n_local, K + 2), dtype=torch.float32, device=dev)
    fl = layer_flops(dims)
    pk = peaks()
    layers_of_exit = np.clip(np.array(model.exit_layers + [dims.layers]), 0, None)

    def sweep_point(conf_thr):
        """all micro-batches of this rank at one threshold; results stay on the device, ONE gather + read-back"""
        thr = thresholds_for(kind, conf_thr, K)
        parts, hist = [], torch.zeros((E1,), dtype=torch.int64, device=dev)
        for d in shards:
            r = model.infer_device(**d, exit_threshold=thr, temperatures=temps)
            parts.append(pack_results(r["logits"], r["exit_index"], r["criterion"]))
            hist += r["hist"]
        packed = torch.cat(parts, dim=0)
        if world > 1:
            dist.all_gather_into_tensor(out_all, packed)
            dist.all_reduce(hist, op=dist.ReduceOp.SUM)
            host = out_all.cpu()
        else:
            host = packed.cpu()
        return host, hist.cpu().numpy()

    for _ in range(max(args.warmup, 3)):                              # warm-up: micro-batch forwards at a mid threshold
        model.infer_device(**shards[0], exit_threshold=thresholds_for(kind, 0.8, K), temperatures=temps)
    torch.cuda.synchronize()
    points = []
    last_steps = []
    with ClockSampler(local, enabled=(rank == 0)) as clk:
        total_ms = 0.0
        for conf_thr in SWEEP_THRESHOLDS:
            ms, (host, hist) = timed_region(lambda: sweep_point(conf_thr), args.steps, 1, world, dev)
            total_ms += ms
            last_steps.append((host, hist))
            reached = reached_per_layer(hist, model.exit_layers, dims.layers, n_total)
            flops = sum(reached) * (fl["linear"] + fl["attn"]) + n_total * fl["patch"]
            tf = flops / (ms / 1000.0) / 1e12
            points.append({"calibrated_confidence_threshold": conf_thr, "docs_per_s": n_total / (ms / 1000.0), "ms": ms,
                           "mean_exit_layer": float(np.dot(hist, layers_of_exit) / hist.sum()),
                           "exit_hist": hist.tolist(), "algorithmic_tflops": tf, "frac_of_tensor_peak": tf / pk["tf_sust"] / world,
                           "predicted_classes_checksum": int(host[:, :K].argmax(1).sum())})
    launches = model.last_launch_count()
    value = n_total * len(SWEEP_THRESHOLDS) / (total_ms / 1000.0)
    if args.dump_outputs and rank == 0:    # per threshold (axis 0): all documents of the job, gathered over the ranks
        out = unpack_results(torch.stack([h for h, _ in last_steps]).numpy(), K)
        out["exit_hist"] = np.stack([hs for _, hs in last_steps])
        dump_outputs(args.dump_outputs, dict(out, temperatures=temps, thresholds=np.array(
            [thresholds_for(kind, t, K) for t in SWEEP_THRESHOLDS])))
    if rank == 0:
        best = max(points, key=lambda p: p["algorithmic_tflops"])
        line = {
            "metric": METRIC, "value": value, "unit": "docs/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype,
            "data": "synthetic",
            "config": {"workload": text, "bench_config": "sweep", "global_batch": n_total, "parallelism": f"dp{world}",
                       "docs_per_gpu": n_local, "micro_batch": MB, "criterion": kind, "thresholds": list(SWEEP_THRESHOLDS),
                       "temperatures": [round(float(t), 5) for t in temps],
                       "l2_policy": "working set per layer (attention bias + activations, several GB) exceeds the 126 MB L2",
                       "step": "one step = all 7 thresholds over all 8192 documents; value = 7 x 8192 / step time"},
            "clocks": clk.summary(), "e2e": None, "gpu_launches": int(launches) * n_mb * len(SWEEP_THRESHOLDS) * args.steps,
            "roofline": {"bound": "tensor", "kernel": "whole hot path (GEMMs + attention) of the documents that reached each layer",
                         "achieved": best["algorithmic_tflops"] / world, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                         "frac": best["frac_of_tensor_peak"], "traffic": None,
                         "note": "per GPU, at the threshold with the deepest exits; per-threshold figures under `sweep`",
                         "peak_source": pk["source"] + " (sustained)"},
            "cpu_baseline": None, "sweep": points,
        }
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
