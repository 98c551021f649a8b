#!/usr/bin/env python
"""Cost of the per-source measurements (cy_measure_sources + cy_measure_combine) on the catalogs of the benchmark
workloads: BASELINE config 3 (16k^2 mosaic, tile step 1.0) and config 4 (32k^2, step 0.5), with bench.py's mosaic,
model and thresholds.  For each: one catalog from pipeline.run_image, then the measurement over the band left in HBM
timed with CUDA events after a warm-up, next to the run_image step time on the same mosaic.  Prints one JSON line per
config with the card name and power limit beside the numbers.

With --noise it also times Engine.measure_noise (all clipping passes, CUDA events around the whole call) and reports
the passes run, the frame bytes each pass reads, the rate over all passes, the share of the run_image step and the
median rms of the catalog next to the noise sigma of synth.make_mosaic.

    python tools/measure_bench.py [--configs 3,4] [--reps 20] [--noise] [--out DIR]
"""
import argparse
import inspect
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (mosaic generator, model and thresholds of the benchmark)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(',')]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:   # the numbers stay meaningful only with the card beside them: say it is unknown
        return {"gpu": "unknown (%s)" % e}


def box_bytes(src, rows, ncols):
    """4-byte pixels the measure kernel reads for the catalog (box area clipped to the image and the owned rows)."""
    x0 = np.maximum(np.ceil(src['x1'].astype(np.float64)), 0)
    x1 = np.minimum(np.floor(src['x2'].astype(np.float64)), ncols - 1)
    y0 = np.maximum(np.ceil(src['y1'].astype(np.float64)), rows[0])
    y1 = np.minimum(np.floor(src['y2'].astype(np.float64)), rows[1] - 1)
    return float((np.clip(x1 - x0 + 1, 0, None) * np.clip(y1 - y0 + 1, 0, None)).sum() * 4)


def frame_pixels(src, rows, ncols, frame):
    """Pixels of each source's frame (grown box minus box, clipped to the image columns and the rows), masked ones
    included: what one noise pass reads for an active source."""
    bx0, bx1 = np.ceil(src['x1'].astype(np.float64)), np.floor(src['x2'].astype(np.float64))
    by0, by1 = np.ceil(src['y1'].astype(np.float64)), np.floor(src['y2'].astype(np.float64))

    def area(x0, x1, y0, y1):
        return np.clip(x1 - x0 + 1, 0, None) * np.clip(y1 - y0 + 1, 0, None)
    gx0, gx1 = np.maximum(bx0 - frame, 0), np.minimum(bx1 + frame, ncols - 1)
    gy0, gy1 = np.maximum(by0 - frame, rows[0]), np.minimum(by1 + frame, rows[1] - 1)
    hole = area(np.maximum(bx0, gx0), np.minimum(bx1, gx1), np.maximum(by0, gy0), np.minimum(by1, gy1))
    return np.where((bx0 <= bx1) & (by0 <= by1), area(gx0, gx1, gy0, gy1) - hole, 0)


def run_noise(eng, src, band, nx, be, Y0, rows, reps, frame, step_ms):
    import torch
    from caesar_yolo_b200 import synth
    for _ in range(2):
        z = eng.measure_noise(src, band, nx, be, Y0, nx, rows[0], rows[1], frame=frame)
    passes = eng.noise_passes
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        eng.measure_noise(src, band, nx, be, Y0, nx, rows[0], rows[1], frame=frame)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    px = frame_pixels(src, rows, nx, frame)
    per_pass = [float(px[z['iters'] >= p].sum() * 4) for p in range(passes)]   # a source is read in passes 0..iters
    ok = z['nbkg'] > 0
    return {"noise_frame": frame, "noise_passes": passes, "frame_bytes_per_pass": per_pass,
            "noise_ms_per_call": round(ms, 4),
            "noise_gbs": round(sum(per_pass) / (ms * 1e-3) / 1e9, 1) if ms > 0 else None,
            "noise_share_of_step": round(ms / step_ms, 5),
            "iters_histogram": np.bincount(z['iters'], minlength=6).tolist(),
            "median_rms": float(np.median(z['rms'][ok])) if ok.any() else None,
            "synth_sigma": inspect.signature(synth.make_mosaic).parameters['sigma'].default,
            "noise_note": "noise_ms_per_call: CUDA events around Engine.measure_noise (catalog upload, unit plan, every "
                          "pass with its host read of the active count, copy of the state back)"}


def run_config(cfg, reps, variant, noise=False, frame=16):
    import torch
    from caesar_yolo_b200 import ops, pipeline, weights as W
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    a = argparse.Namespace(mosaic=32768 if cfg == 4 else 16384)
    step = 0.5 if cfg == 4 else 1.0
    n = a.mosaic
    _, host = bench.make_mosaic_pinned(a)
    tiles = ops.generate_tiles(0, n - 1, 0, n - 1, 512, 512, step, step)
    w = W.make_random_weights(variant, 5, seed=0, cls_bias=bench.CLS_BIAS.get(variant, -16.0))
    eng = pipeline.Engine(w, pipeline.make_pp_config(**bench.PP_FLAGS), imgsz=640, score_thr=bench.SCORE_THR,
                          iou_thr=bench.IOU_THR, thr_soft=bench.SOFT, thr_hard=bench.HARD, device=dev)

    def step_fn():
        return pipeline.run_image(eng, host, True, tiles)

    step_fn()                                           # warm-up (plans, buffers)
    torch.cuda.synchronize()
    t0 = time.time()
    k = 2
    for _ in range(k):
        src, _ = step_fn()
    torch.cuda.synchronize()
    step_ms = (time.time() - t0) * 1e3 / k
    band, Y0, _, nx, be = eng.band
    r0, r1 = pipeline.measure_rows(tiles, 1)[0]
    src_dev = ops.to_device_bytes(np.ascontiguousarray(src), dev)
    ns = len(src)
    part = torch.empty((ns * ops.PARTIAL_BYTES,), dtype=torch.uint8, device=dev)
    meas = torch.empty((ns * ops.MEAS_DTYPE.itemsize,), dtype=torch.uint8, device=dev)

    def measure():
        ops.measure_sources(band, nx, be, Y0, nx, src_dev, ns, r0, r1, out=part)
        ops.measure_combine(part, 1, src_dev, ns, nx, out=meas)

    for _ in range(3):
        measure()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        measure()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # Engine.measure as SFinder calls it (upload of the catalog, kernels, copy of the results to the host)
    torch.cuda.synchronize()
    t0 = time.time()
    for _ in range(reps):
        eng.measure(src, band, nx, be, Y0, nx, r0, r1)
    torch.cuda.synchronize()
    engine_ms = (time.time() - t0) * 1e3 / reps
    nbytes = box_bytes(src, (r0, r1), nx)
    r = {"config": cfg, "mosaic": n, "tile_step": step, "tiles": len(tiles), "sources": ns,
         "measure_ms_per_call": round(ms, 4), "engine_measure_ms_per_call": round(engine_ms, 4),
         "box_bytes_read": nbytes, "box_gbs": round(nbytes / (ms * 1e-3) / 1e9, 1) if ms > 0 else None,
         "run_image_step_ms": round(step_ms, 2), "measure_share_of_step": round(engine_ms / step_ms, 5),
         "note": "measure_ms_per_call: CUDA events around cy_measure_sources + cy_measure_combine (includes the "
                 "one host read of the unit count); the band stays resident in L2 only in part (16k^2 band = 1 GB)"}
    if noise:
        r.update(run_noise(eng, src, band, nx, be, Y0, (r0, r1), reps, frame, step_ms))
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='3,4')
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--variant', default='l')
    ap.add_argument('--noise', action='store_true', help='also time the local background / noise passes')
    ap.add_argument('--noise_frame', type=int, default=16)
    ap.add_argument('--out', default=None, help='directory for measure_bench.json')
    a = ap.parse_args()
    info = card()
    lines = []
    for c in [int(x) for x in a.configs.split(',')]:
        r = run_config(c, a.reps, a.variant, a.noise, a.noise_frame)
        r.update(info)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'measure_bench.json'), 'w') as f:
            json.dump(lines, f, indent=1)


if __name__ == '__main__':
    main()
