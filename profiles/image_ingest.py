"""Cost of getting document images into the engine: the host LayoutLMv3 image processor vs the device preprocess.

    python profiles/image_ingest.py --out DIR [--batch 256] [--reps 200] [--e2e-rounds 4]

Headline configuration of bench.py (LayoutLMv3-base, concat exit + gates after all 12 layers, entropy policy with
calibrated temperatures), B = 256 documents per call.  Pages are seeded synthetic grayscale scans: height 1000, width
uniform in [600, 1000], dark text-like stripes on a light background plus noise (RVL-CDIP-shaped).  Measured:

  host_processor   transformers' LayoutLMv3ImageProcessorPil(apply_ocr=False) per page, on one thread and with one
                   worker process per host core (wall time / pages)
  device           model.preprocess_images on 256 resident uint8 pages: CUDA events, warmed up, --reps repetitions
  e2e (docs/s)     (a) infer(pixel_values = host fp32, prepared beforehand)  engine only
                   (b) infer(images = packed uint8 pages, pinned)          upload + device preprocess + engine
                   (c) host processor on all cores, then (a)               what a caller without (b) runs
                   (a) and (b) alternate in rounds; (c) runs fewer batches (it is slow)

Also written: upload bytes per page of (a) and (b), whether the device pixels equal the host processor's bit for bit on
every page, and the card's name, power limit and max SM clock read in the same run.  Writes DIR/image_ingest.json.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "multi-modal-early-exit_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from latency import card  # noqa: E402
from mmee import synth  # noqa: E402
from mmee.calibration import thresholds_for  # noqa: E402
from mmee.images import pack_images  # noqa: E402


def make_pages(n, seed):
    """Seeded grayscale pages, 1000 x U{600..1000}: text-like stripes (dark runs on light rows) and noise."""
    rng = np.random.default_rng(seed)
    pages = []
    for _ in range(n):
        h, w = 1000, int(rng.integers(600, 1001))
        a = np.full((h, w), 235, np.int16)
        line_h = int(rng.integers(10, 20))
        for y in range(int(rng.integers(40, 80)), h - 60, int(line_h * rng.uniform(1.6, 2.4))):
            x = int(rng.integers(40, 80))
            while x < w - 60:
                run = int(rng.integers(5, 60))
                a[y:y + line_h, x:min(x + run, w - 60)] = int(rng.integers(10, 80))
                x += run + int(rng.integers(4, 12))
        a += rng.normal(0, 12, (h, w)).astype(np.int16)
        pages.append(np.clip(a, 0, 255).astype(np.uint8))
    return pages


_proc = None


def _init_worker():
    global _proc
    from transformers import LayoutLMv3ImageProcessorPil

    _proc = LayoutLMv3ImageProcessorPil(apply_ocr=False)


def host_process(a):
    """The reference's host path for one decoded page: PIL image, convert("RGB"), processor -> f32 [3, 224, 224]."""
    from PIL import Image

    return _proc(Image.fromarray(a).convert("RGB"), return_tensors="np")["pixel_values"][0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--e2e-rounds", type=int, default=4)
    ap.add_argument("--host-pages", type=int, default=64, help="pages timed through the processor on one thread")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("image_ingest.py measures the GPU: no CUDA device")
    from mmee.model import B200EEForSequenceClassification

    B = args.batch
    cores = os.cpu_count()
    result = {"card": card(), "batch": B, "host_cores": cores,
              "pages": "grayscale 1000 x U{600..1000}, text-like stripes + noise (seeded)"}
    print(json.dumps(result["card"]), flush=True)
    pages = make_pages(B, seed=7)

    # host processor: one thread, then one worker per core
    _init_worker()
    for a in pages[:4]:
        host_process(a)
    t0 = time.perf_counter()
    for a in pages[:args.host_pages]:
        host_process(a)
    one = (time.perf_counter() - t0) / args.host_pages
    with mp.get_context("fork").Pool(cores, initializer=_init_worker) as pool:
        pool.map(host_process, pages[:cores])                       # workers up
        t0 = time.perf_counter()
        host_px = np.stack(pool.map(host_process, pages, chunksize=max(B // (4 * cores), 1)))
        allc = (time.perf_counter() - t0) / B
        result["host_processor"] = {"ms_per_page_one_thread": one * 1e3, "ms_per_page_all_cores": allc * 1e3,
                                    "pages_per_s_all_cores": 1.0 / allc}
        print(json.dumps(result["host_processor"]), flush=True)

        dims, ee, _, text, dtype = bench.workload("headline")
        sd = synth.make_state_dict(dims, ee, seed=0)
        model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=B, dtype=dtype)
        dev = torch.device("cuda", 0)
        kind = ee.inference_strategy
        temps = bench.calibrate_temperatures(model, dims, kind, dev)
        kw = dict(exit_threshold=thresholds_for(kind, bench.CONF_THRESHOLD, dims.n_labels), temperatures=temps)

        # device preprocess of B resident pages
        packed = pack_images(pages)
        resident = pack_images(pages, pin=True)
        resident.data = resident.data.to(dev)
        px_dev = model.preprocess_images(resident)
        torch.cuda.synchronize()
        result["device_equals_host_processor"] = bool(np.array_equal(px_dev.cpu().numpy(), host_px))
        for _ in range(20):
            model.preprocess_images(resident)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(args.reps):
            model.preprocess_images(resident)
        ev[1].record()
        torch.cuda.synchronize()
        dev_ms = ev[0].elapsed_time(ev[1]) / args.reps
        result["device_preprocess"] = {"ms_per_batch": dev_ms, "us_per_page": dev_ms * 1e3 / B, "reps": args.reps,
                                       "bytes_read": int(resident.data.numel())}
        print(json.dumps(result["device_preprocess"]), flush=True)

        # end to end
        docs = synth.make_docs(dims, B, seed=11, pad=False)
        txt = {k: v.pin_memory() for k, v in docs.items() if k != "pixel_values"}
        px_host = torch.from_numpy(host_px).pin_memory()
        run = {"a_pixel_values": lambda: model.infer(**txt, pixel_values=px_host, **kw),
               "b_images": lambda: model.infer(**txt, images=packed, **kw)}
        ra, rb = run["a_pixel_values"](), run["b_images"]()
        result["e2e_b_equals_a"] = bool(torch.equal(ra.logits, rb.logits) and np.array_equal(ra.exits_store, rb.exits_store))
        for f in run.values():
            for _ in range(3):
                f()
        times = {k: [] for k in run}
        for _ in range(args.e2e_rounds):
            for k, f in run.items():
                for _ in range(5):
                    t0 = time.perf_counter()
                    f()
                    times[k].append(time.perf_counter() - t0)
        times["c_host_processor_then_a"] = []
        for _ in range(3):
            t0 = time.perf_counter()
            px = torch.from_numpy(np.stack(pool.map(host_process, pages, chunksize=max(B // (4 * cores), 1))))
            model.infer(**txt, pixel_values=px, **kw)
            times["c_host_processor_then_a"].append(time.perf_counter() - t0)
    result["e2e"] = {k: {"docs_per_s": float(B / np.mean(t)), "ms_per_batch_mean": float(np.mean(t) * 1e3),
                         "ms_per_batch_min": float(np.min(t) * 1e3), "batches": len(t)} for k, t in times.items()}
    result["upload_bytes_per_page"] = {"a_pixel_values": 3 * dims.image * dims.image * 4,
                                       "b_images": float(packed.data.numel() / B)}
    result["card_after"] = card()
    print(json.dumps({"e2e": result["e2e"], "upload": result["upload_bytes_per_page"],
                      "device_equals_host_processor": result["device_equals_host_processor"],
                      "e2e_b_equals_a": result["e2e_b_equals_a"]}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "image_ingest.json"), "w") as f:
        json.dump(result, f, indent=1)
    if not (result["device_equals_host_processor"] and result["e2e_b_equals_a"]):
        raise SystemExit("device preprocess differs from the host processor")


if __name__ == "__main__":
    main()
