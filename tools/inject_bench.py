#!/usr/bin/env python
"""Cost of one source-injection round (inject.run_rounds, the steps of SFinder with inject_sources) on the benchmark
workloads: BASELINE config 3 (16k^2 mosaic, tile step 1.0) and config 4 (32k^2, step 0.5), with bench.py's mosaic,
model and thresholds, at the default bkg box and grid, with N = 1024 and 4096 injections per round.  For each config:
one pipeline.run_image (the band stays in HBM) after a warm-up, timed on the host clock around a device synchronise (the
detection step), then the node states without map rows (Engine.bkg_maps_band with maps=False), then --rounds rounds per
N.  Every step of a round ends with a device synchronise and is timed on the host clock:
  sample_s   cy_bkg_grid_sample of the rms at every candidate centre (one call per round, copy to the host included)
  place_s    the host placement, sampling excluded
  inject_s   cy_inject_sources (saved words included)
  rerun_s    Engine.process_tiles of the affected tiles (their count is reported)
  merge_s    Engine.exchange_and_merge (one rank: compaction and cross-tile merge)
  restore_s  cy_inject_restore and the copy of the record snapshot
The card name and power limit are read in the same call and written beside the numbers.

    python tools/inject_bench.py [--configs 3,4] [--n 1024,4096] [--rounds 2] [--out DIR]
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

WCS = {"BMAJ": 0.0025, "BMIN": 0.002, "BPA": 30.0, "CDELT1": -0.0004, "CDELT2": 0.0004}   # the synthetic mosaic's beam


def run_config(cfg, ns, rounds, variant, box, grid):
    import torch
    from caesar_yolo_b200 import fits, inject, ops, pipeline, weights as W
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
    pipeline.run_image(eng, host, True, tiles)          # warm-up (plans, buffers)
    torch.cuda.synchronize()
    t0 = time.time()
    src, _ = pipeline.run_image(eng, host, True, tiles)
    torch.cuda.synchronize()
    step_s = time.time() - t0
    t0 = time.time()
    nodes = eng.bkg_maps_band(tiles, box, grid, maps=False)[0]
    nodes_s = time.time() - t0
    words = host.numpy().view(np.uint32)

    def centre_masked(cx, cy):
        v = words[cy, cx].byteswap().view(np.float32)
        return ~np.isfinite(v) | (v == 0)
    cov = fits.beam_cov_pix(WCS)
    bx0, bx1, by0, by1 = inject.integer_boxes(src)
    area = np.maximum(bx1 - bx0 + 1, 0) * np.maximum(by1 - by0 + 1, 0)
    out = {"config": cfg, "mosaic": n, "tile_step": step, "tiles": int(len(tiles)), "catalog_sources": int(len(src)),
           "catalog_box_area_sum_over_image": round(float(area.sum()) / (n * n), 4),
           "catalog_largest_box_over_image": round(float(area.max()) / (n * n), 4) if len(area) else 0.0,
           "bkg_box": box, "bkg_grid": grid, "footprint_half": list(inject.footprint_half(cov)),
           "detection_step_s": round(step_s, 4), "node_states_s": round(nodes_s, 4), "per_n": []}
    for N in ns:
        plan = inject.tiled_plan(eng, tiles, src, nodes, box, grid, centre_masked)
        sample = {'s': 0.0}
        real = plan.sample_rms

        def timed_sample(cx, cy, real=real, sample=sample):
            t = time.time()
            r = real(cx, cy)
            sample['s'] += time.time() - t
            return r
        plan.sample_rms = timed_sample
        inject.run_rounds(eng, plan, N, 1, (3.0, 100.0), 0, cov, eng.names)   # warm-up of the shapes
        sample['s'] = 0.0
        timing = {}
        res = inject.run_rounds(eng, plan, N, rounds, (3.0, 100.0), 1, cov, eng.names, timing=timing)
        per = {k: round(v / rounds, 4) for k, v in timing.items() if k.endswith('_s')}
        per['sample_s'] = round(sample['s'] / rounds, 4)
        per['place_s'] = round((timing['place_s'] - sample['s']) / rounds, 4)
        per['round_s'] = round(sum(v for k, v in timing.items() if k.endswith('_s')) / rounds, 4)
        placed = [r['placed'] for r in res[1]]
        rec = sum(d['recovered'] for d in res[0])
        rej = {k: sum(r['rejected'][k] for r in res[1]) for k in inject.REJECT_RULES}
        out["per_n"].append(dict(n=N, rounds=rounds, placed=placed, recovered=int(rec), rejected=rej,
                                 affected_tiles=int(timing['affected_tiles'] // rounds),
                                 round_over_detection_step=round(per['round_s'] / step_s, 3), **per))
    out["note"] = ("host clock around each step, each ending with a device synchronise; sample_s is the rms sampling "
                   "call inside the placement (subtracted from place_s); averages over the timed rounds after one "
                   "warm-up round per N; one rank")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='3,4')
    ap.add_argument('--n', default='1024,4096')
    ap.add_argument('--rounds', type=int, default=2)
    ap.add_argument('--variant', default='l')
    ap.add_argument('--bkg_box', type=int, default=101)
    ap.add_argument('--bkg_grid', type=int, default=25)
    ap.add_argument('--out', default=None, help='directory for r08_inject_bench.json')
    a = ap.parse_args()
    info = card()
    res = []
    for c in [int(x) for x in a.configs.split(',')]:
        r = run_config(c, [int(x) for x in a.n.split(',')], a.rounds, a.variant, a.bkg_box, a.bkg_grid)
        r.update(info)
        print(json.dumps(r), flush=True)
        res.append(r)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'r08_inject_bench.json'), 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
