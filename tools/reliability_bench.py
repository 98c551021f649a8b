#!/usr/bin/env python
"""Cost of the reliability estimate (reliability.run, the steps of SFinder with reliability) on the benchmark
workloads: BASELINE config 3 (16k^2 mosaic, tile step 1.0) and config 4 (32k^2, step 0.5), with bench.py's mosaic,
model and thresholds, at the default bkg box and grid, on one GPU.  For each config: one pipeline.run_image (the band
stays in HBM) after a warm-up, timed on the host clock around a device synchronise (the detection step), then the node
states without map rows (Engine.bkg_maps_band with maps=False), then one warm-up run and --repeats timed runs of
reliability.run.  Every step ends with a device synchronise and is timed on the host clock:
  negate_s               cy_negate_rows over the band (the record snapshot included)
  rerun_s                Engine.process_tiles of every tile
  merge_s                Engine.exchange_and_merge (one rank: compaction and cross-tile merge)
  restore_s              the copy of the record snapshot and cy_negate_rows again
  peak_snr_catalog_s     cy_source_peak_snr of the catalog (copies to and from the host included)
  peak_snr_negative_s    the same for the negative catalog
The card name and power limit are read in the same call and written beside the numbers.

    python tools/reliability_bench.py [--configs 3,4] [--repeats 2] [--out DIR]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (mosaic generator, model and thresholds of the benchmark)
from measure_bench import card  # noqa: E402


def run_config(cfg, repeats, variant, box, grid):
    import torch
    from caesar_yolo_b200 import inject, ops, pipeline, reliability, weights as W
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
    pipeline.run_image(eng, host, True, tiles, on_rank0_only=False)          # warm-up (plans, buffers)
    torch.cuda.synchronize()
    t0 = time.time()
    src, _ = pipeline.run_image(eng, host, True, tiles, on_rank0_only=False)
    torch.cuda.synchronize()
    step_s = time.time() - t0
    t0 = time.time()
    nodes = eng.bkg_maps_band(tiles, box, grid, maps=False)[0]
    nodes_s = time.time() - t0
    band = eng.band[0]
    before = band.clone()
    plan = reliability.tiled_plan(eng, tiles, src, nodes, box, grid)
    neg, pos_peak, neg_peak = reliability.run(eng, plan)                    # warm-up of the shapes
    timing = {}
    for _ in range(repeats):
        neg, pos_peak, neg_peak = reliability.run(eng, plan, timing=timing)
    torch.cuda.synchronize()
    restored = bool(torch.equal(band, before))
    del before
    per = {k: round(v / repeats, 4) for k, v in timing.items()}
    per['total_s'] = round(sum(timing.values()) / repeats, 4)
    bx0, bx1, by0, by1 = inject.integer_boxes(src)
    area = np.maximum(bx1 - bx0 + 1, 0) * np.maximum(by1 - by0 + 1, 0)
    band_bytes = int(band.numel()) * 4
    out = {"config": cfg, "mosaic": n, "tile_step": step, "tiles": int(len(tiles)), "catalog_sources": int(len(src)),
           "negative_sources": int(len(neg)), "catalog_box_pixels": int(area.sum()),
           "catalog_peak_snr_nan": int(np.isnan(pos_peak[0]).sum()),
           "negative_peak_snr_nan": int(np.isnan(neg_peak[0]).sum()),
           "bkg_box": box, "bkg_grid": grid, "band_bytes": band_bytes, "rows_restored_bit_for_bit": restored,
           "detection_step_s": round(step_s, 4), "node_states_s": round(nodes_s, 4), "repeats": repeats,
           "total_over_detection_step": round(per['total_s'] / step_s, 3), **per}
    out["note"] = ("host clock around each step, each ending with a device synchronise; averages over the timed runs "
                   "after one warm-up run; one rank; the band is negated in place (8 bytes of traffic per pixel per "
                   "call, two calls per run)")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='3,4')
    ap.add_argument('--repeats', type=int, default=2)
    ap.add_argument('--variant', default='l')
    ap.add_argument('--bkg_box', type=int, default=101)
    ap.add_argument('--bkg_grid', type=int, default=25)
    ap.add_argument('--out', default=None, help='directory for r09_reliability_bench.json')
    a = ap.parse_args()
    info = card()
    res = []
    for c in [int(x) for x in a.configs.split(',')]:
        r = run_config(c, a.repeats, a.variant, a.bkg_box, a.bkg_grid)
        r.update(info)
        print(json.dumps(r), flush=True)
        res.append(r)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'r09_reliability_bench.json'), 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
