#!/usr/bin/env python
"""Cost of the background / rms maps (Engine.bkg_maps: cy_bkg_grid_init, the clipping passes, cy_bkg_grid_maps) on the
benchmark workloads: BASELINE config 3 (16k^2 mosaic, tile step 1.0) and config 4 (32k^2, step 0.5), with bench.py's
mosaic, model and thresholds, at the default box and grid.  For each: one pipeline.run_image (the band stays in HBM),
then Engine.bkg_maps_band timed with CUDA events after a warm-up, next to the run_image step time on the same mosaic;
each clipping pass is timed on its own with events; the two map files are written once with fits.write_map_rows and
timed on the host clock.  Prints one JSON line per config with the card name and power limit beside the numbers.

Algorithmic bytes of pass p: for every unit whose node group has an active node in pass p, the 4-byte pixels of its
rows and of the columns from its first to its last active node's box (what bkg_unit_kernel reads), plus the unit
partials written and folded.  The map kernel writes 8 bytes per pixel and reads no image pixel.

With --mask, the source mask is timed as well on the catalog of the same run_image: the mask build
(Engine.source_mask_band), the masked map call (Engine.bkg_maps_band with the mask: masked passes, probe and fill), the
probe and fill alone (events around cy_bkg_grid_probe_init, the probe pass and cy_bkg_grid_fill, restated from the final
masked states), and the local noise of the catalog with and without the mask (Engine.measure_noise_band).  The masked and
unmasked calls alternate within each repetition, so both see the same machine state.  It reports the masked pixel
fraction, the nodes left without pixels and the holes filled, and writes r05_bkgmask_bench.json to --out.

With --estimator median, the median estimator is timed against the mean on the catalog of the same run_image:
Engine.measure_noise_band and Engine.bkg_maps_band, each unmasked and with the source mask, the median and the mean
calls alternating within each repetition.  It reports the pass counts, the bytes of the select histograms and how far
the median and mean node bkg lie apart, and writes r06_bkgmedian_bench.json to --out.

With --snr, the background-subtracted and S/N maps are timed from the final node states of the same run_image's band:
cy_bkg_grid_snr_maps alone (CUDA events around --reps launches into preallocated rows, after a warm-up; the 12 bytes per
pixel of a 16k^2 or 32k^2 region are far more than the 126 MB L2, so every launch reads and writes HBM), alternating with
cy_bkg_grid_maps into the same kind of rows, and the Engine.snr_maps_band call (row allocation and node upload included).
Algorithmic bytes: 4 read and 8 written per pixel, plus the bkg and rms of every node once.  The two files are written
once and timed on the host clock.  Writes r07_snrmap_bench.json to --out.

    python tools/bkgmap_bench.py [--configs 3,4] [--reps 5] [--mask | --estimator median | --snr] [--out DIR]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (mosaic generator, model and thresholds of the benchmark)
from measure_bench import card  # noqa: E402

GROUP, UNIT_ROWS, PARTIAL = 16, 32, 24


def pass_bytes(nodes, W, H, box, grid):
    """Bytes each pass reads / writes (module docstring), from the final node states: node n is active in passes
    0 .. iters[n] (an empty node stops after pass 0)."""
    from caesar_yolo_b200 import ops
    h = box // 2
    xs, ys = np.array(ops.bkg_grid_nodes(W, grid)), np.array(ops.bkg_grid_nodes(H, grid))
    out = []
    for p in range(int(nodes['iters'].max()) + 1):
        act = nodes['iters'] >= p
        total = 0
        for j, y in enumerate(ys):
            rows = min(y + h, H - 1) - max(y - h, 0) + 1
            nch = (rows - 1) // UNIT_ROWS + 1
            for g0 in range(0, len(xs), GROUP):
                a = np.nonzero(act[j, g0:g0 + GROUP])[0]
                if a.size == 0:
                    continue
                cols = min(xs[g0 + a[-1]] + h, W - 1) - max(xs[g0 + a[0]] - h, 0) + 1
                total += rows * cols * 4 + nch * GROUP * PARTIAL * 2
        out.append(float(total))
    return out


def run_config(cfg, reps, variant, box, grid):
    import torch
    from caesar_yolo_b200 import fits, ops, pipeline, weights as W
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
    k = 2
    for _ in range(k):
        src, _ = pipeline.run_image(eng, host, True, tiles)
    torch.cuda.synchronize()
    step_ms = (time.time() - t0) * 1e3 / k
    res = None
    for _ in range(2):
        res = eng.bkg_maps_band(tiles, box, grid)
    nodes, bkg, rms, (X0, R0, Wd, Hd), rows = res
    passes = eng.bkg_passes
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        eng.bkg_maps_band(tiles, box, grid)
    e1.record()
    torch.cuda.synchronize()
    call_ms = e0.elapsed_time(e1) / reps
    # every pass on its own: the engine's loop restated with events around each cy_bkg_grid_pass
    band, Y0, _, nx, be = eng.band
    img = band[:, X0:]
    nn = nodes.size
    state = torch.empty((nn * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
    off = torch.empty((nodes.shape[0] + 1,), dtype=torch.int64, device=dev)
    part = torch.empty((nn * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev)
    pass_ms = [0.0] * passes
    for _ in range(reps):
        units = ops.bkg_grid_init(Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, state, off)
        for p in range(passes):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            ops.bkg_grid_pass(img, nx, be, Y0, Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, off, units, state, part)
            a1.record()
            ops.noise_update(part, 1, nn, state)
            pass_ms[p] += a0.elapsed_time(a1) / reps
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record()
    for _ in range(reps):
        ops.bkg_grid_maps(state, Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, bkg, rms)
    m1.record()
    torch.cuda.synchronize()
    map_ms = m0.elapsed_time(m1) / reps
    nbytes = pass_bytes(nodes, Wd, Hd, box, grid)
    with tempfile.TemporaryDirectory() as d:
        hdr = fits.map_header({}, Wd, Hd, X0, R0)
        t0 = time.time()
        for name, m in (('bkgmap.fits', bkg), ('rmsmap.fits', rms)):
            fits.write_map_rows(os.path.join(d, name), hdr, m, 0, Wd, Hd)
        write_s = time.time() - t0
    ok = nodes['nbkg'] > 0
    return {"config": cfg, "mosaic": n, "tile_step": step, "bkg_box": box, "bkg_grid": grid,
            "nodes": [int(nodes.shape[0]), int(nodes.shape[1])], "passes": passes,
            "iters_histogram": np.bincount(nodes['iters'].ravel(), minlength=6).tolist(),
            "bkg_maps_ms_per_call": round(call_ms, 3), "pass_ms": [round(x, 3) for x in pass_ms],
            "map_rows_ms": round(map_ms, 3),
            "pass_bytes": nbytes, "pass_gbs": [round(b / (t * 1e-3) / 1e9, 1) if t > 0 else None
                                               for b, t in zip(nbytes, pass_ms)],
            "map_bytes_written": 8 * Wd * Hd,
            "run_image_step_ms": round(step_ms, 2), "bkg_maps_share_of_step": round(call_ms / step_ms, 4),
            "file_write_s": round(write_s, 3), "file_bytes": 2 * (len(hdr) + 4 * Wd * Hd),
            "median_node_rms": float(np.median(nodes['rms'][ok])) if ok.any() else None,
            "note": "bkg_maps_ms_per_call: CUDA events around Engine.bkg_maps_band (unit plan, every pass with its host "
                    "read of the active count, map rows, copy of the node states to the host); pass_ms: events around "
                    "cy_bkg_grid_pass alone; file_write_s: host clock around both files (device -> pinned -> pwrite, "
                    "one rank, a temporary directory on the local disk)"}


def _events(fn, reps):
    """ms per call of fn over reps calls, CUDA events around each call (fn synchronises inside: host reads)."""
    import torch
    t = 0.0
    for _ in range(reps):
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        fn()
        a1.record()
        torch.cuda.synchronize()
        t += a0.elapsed_time(a1)
    return t / reps


def mask_config(cfg, reps, variant, box, grid, frame=16):
    """The --mask measurements of one config (module docstring)."""
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
    src, _ = pipeline.run_image(eng, host, True, tiles)
    mask = eng.source_mask_band(src, tiles)              # warm-up of every call timed below
    plain = eng.bkg_maps_band(tiles, box, grid)[0]
    nodes, _, _, (X0, R0, Wd, Hd), rows = eng.bkg_maps_band(tiles, box, grid, mask=mask)
    passes, filled = eng.bkg_passes, eng.bkg_holes_filled
    eng.measure_noise_band(src, tiles, frame)
    eng.measure_noise_band(src, tiles, frame, mask=mask)
    ms = dict(mask=0.0, maps=0.0, maps_masked=0.0, noise=0.0, noise_masked=0.0)
    for _ in range(reps):                                # the masked and unmasked calls alternate
        ms['mask'] += _events(lambda: eng.source_mask_band(src, tiles), 1) / reps
        ms['maps'] += _events(lambda: eng.bkg_maps_band(tiles, box, grid), 1) / reps
        ms['maps_masked'] += _events(lambda: eng.bkg_maps_band(tiles, box, grid, mask=mask), 1) / reps
        ms['noise'] += _events(lambda: eng.measure_noise_band(src, tiles, frame), 1) / reps
        ms['noise_masked'] += _events(lambda: eng.measure_noise_band(src, tiles, frame, mask=mask), 1) / reps
    noise_passes = eng.noise_passes
    # probe and fill alone, from the final masked states (restated: the masked passes, then a copy of the states)
    band, Y0, _, nx, be = eng.band
    img = band[:, X0:]
    nn = nodes.size
    state = torch.empty((nn * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
    probe = torch.empty_like(state)
    off = torch.empty((nodes.shape[0] + 1,), dtype=torch.int64, device=dev)
    part = torch.empty((nn * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev)
    units = ops.bkg_grid_init(Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, state, off)
    active = nn
    while active:
        ops.bkg_grid_pass_masked(img, nx, be, Y0, Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, off, units, state, part,
                                 mask.bits, mask.ncols, X0)
        active = ops.noise_update(part, 1, nn, state)
    saved = state.clone()

    def probe_fill():
        state.copy_(saved)
        if ops.bkg_grid_probe_init(state, nn, probe):
            ops.bkg_grid_pass(img, nx, be, Y0, Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, off, units, probe, part)
            ops.bkg_grid_fill(part, 1, nodes.shape[1], nodes.shape[0], state)
    probe_fill()
    probe_ms = _events(probe_fill, reps)
    assert state.cpu().numpy().view(ops.NOISE_DTYPE).tobytes() == nodes.tobytes()
    mbits = 0
    mh = mask.bits.cpu().numpy().view(np.uint8)
    for r in range(0, mh.shape[0], 1024):
        mbits += int(np.unpackbits(mh[r:r + 1024]).sum())
    masked_frac = mbits / float(mh.shape[0] * nx)
    return {"config": cfg, "mosaic": n, "tile_step": step, "bkg_box": box, "bkg_grid": grid, "noise_frame": frame,
            "sources": int(len(src)), "masked_pixel_fraction": round(masked_frac, 5),
            "nodes": [int(nodes.shape[0]), int(nodes.shape[1])], "passes_masked": passes,
            "nodes_without_pixels_unmasked": int(np.sum(plain['nbkg'] == 0)),
            "nodes_without_pixels_masked": int(np.sum(nodes['nbkg'] == 0)), "holes_filled": int(filled),
            "noise_passes": noise_passes,
            "source_mask_ms": round(ms['mask'], 3), "bkg_maps_ms": round(ms['maps'], 3),
            "bkg_maps_masked_ms": round(ms['maps_masked'], 3), "probe_fill_ms": round(probe_ms, 3),
            "noise_ms": round(ms['noise'], 3), "noise_masked_ms": round(ms['noise_masked'], 3),
            "note": "CUDA events around each call, synchronised after it; the masked and unmasked calls alternate in "
                    "every repetition.  bkg_maps_masked_ms includes the masked passes, the probe and the fill, not the "
                    "mask build (source_mask_ms, built once per run); probe_fill_ms: cy_bkg_grid_probe_init, the probe "
                    "pass and cy_bkg_grid_fill from the final masked states"}


def median_config(cfg, reps, variant, box, grid, frame=16):
    """The --estimator median measurements of one config (module docstring)."""
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
    src, _ = pipeline.run_image(eng, host, True, tiles)
    mask = eng.source_mask_band(src, tiles)
    calls = {}
    for est in ('mean', 'median'):
        for m in (None, mask):
            tag = est + ('_masked' if m is not None else '')
            calls['noise_' + tag] = (lambda e=est, mm=m: eng.measure_noise_band(src, tiles, frame, mask=mm,
                                                                                estimator=e))
            calls['maps_' + tag] = (lambda e=est, mm=m: eng.bkg_maps_band(tiles, box, grid, mask=mm, estimator=e))
    out, passes = {}, {}
    for k, fn in calls.items():                          # warm-up of every call timed below
        out[k] = fn()
        passes[k] = eng.noise_passes if k.startswith('noise') else eng.bkg_passes
    ms = {k: 0.0 for k in calls}
    for _ in range(reps):                                # the median and mean calls alternate
        for k, fn in calls.items():
            ms[k] += _events(fn, 1) / reps
    nodes_mean, nodes_med = out['maps_mean'][0], out['maps_median'][0]
    ok = (nodes_mean['nbkg'] > 0) & (nodes_med['nbkg'] > 0)
    dz = np.abs(nodes_med['bkg'][ok] - nodes_mean['bkg'][ok]) / nodes_mean['rms'][ok]
    return {"config": cfg, "mosaic": n, "tile_step": step, "bkg_box": box, "bkg_grid": grid, "noise_frame": frame,
            "sources": int(len(src)), "nodes": [int(nodes_med.shape[0]), int(nodes_med.shape[1])],
            "passes": passes, "ms": {k: round(v, 3) for k, v in ms.items()},
            "median_over_mean": {k: round(ms[k.replace('mean', 'median')] / ms[k], 2) for k in ms if 'mean' in k},
            "select_histogram_bytes": {"noise": len(src) * ops.SELECT_SLOTS * 4,
                                       "maps": int(nodes_med.size) * ops.SELECT_SLOTS * 4},
            "node_bkg_median_minus_mean_over_rms": {"median": float(np.median(dz)), "max": float(dz.max())},
            "note": "CUDA events around each call, synchronised after it (Engine.measure_noise_band / bkg_maps_band: "
                    "unit plan, every pass with its host read of the active count; the median passes are 4 digit "
                    "rounds each); the median and mean calls alternate in every repetition; the masked calls include "
                    "the probe and fill of the maps, not the mask build (built once)"}


def snr_config(cfg, reps, variant, box, grid):
    """The --snr measurements of one config (module docstring)."""
    import torch
    from caesar_yolo_b200 import fits, ops, pipeline, weights as W
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
    pipeline.run_image(eng, host, True, tiles)
    nodes, bkg, rms, (X0, R0, Wd, Hd), rows = eng.bkg_maps_band(tiles, box, grid)
    res, snr, _, _ = eng.snr_maps_band(nodes, tiles, box, grid)          # warm-up of the Engine call
    band, Y0, _, nx, be = eng.band
    img = band[:, X0:]
    state = ops.to_device_bytes(nodes, dev)
    res2, snr2 = torch.empty_like(res), torch.empty_like(snr)

    def snr_call():
        ops.bkg_grid_snr_maps(state, img, nx, be, Y0, Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, res2, snr2)

    def map_call():
        ops.bkg_grid_maps(state, Wd, R0, R0 + Hd, rows[0], rows[1], box, grid, bkg, rms)
    snr_call()
    map_call()
    torch.cuda.synchronize()
    same = bool(torch.equal(res, res2) and torch.equal(snr, snr2))
    ms = dict(snr=0.0, maps=0.0, engine=0.0)
    for _ in range(reps):                                # the two kernels alternate, reps launches each
        for k, fn in (('snr', snr_call), ('maps', map_call)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms[k] += e0.elapsed_time(e1) / (reps * reps)
        ms['engine'] += _events(lambda: eng.snr_maps_band(nodes, tiles, box, grid), 1) / reps
    pix = Wd * (rows[1] - rows[0])
    snr_bytes = 12 * pix + 16 * nodes.size
    with tempfile.TemporaryDirectory() as d:
        t0 = time.time()
        for name, m, unit in (('resmap.fits', res, True), ('snrmap.fits', snr, False)):
            fits.write_map_rows(os.path.join(d, name), fits.map_header({}, Wd, Hd, X0, R0, bunit=unit), m, 0, Wd, Hd)
        write_s = time.time() - t0
    f = snr.cpu().numpy().view('>f4')
    finite = float(np.isfinite(f).mean())
    return {"config": cfg, "mosaic": n, "tile_step": step, "bkg_box": box, "bkg_grid": grid,
            "nodes": [int(nodes.shape[0]), int(nodes.shape[1])], "pixels": pix,
            "snr_kernel_ms": round(ms['snr'], 3), "snr_bytes": snr_bytes,
            "snr_tb_s": round(snr_bytes / (ms['snr'] * 1e-3) / 1e12, 2),
            "bkg_map_kernel_ms": round(ms['maps'], 3), "bkg_map_bytes": 8 * pix + 16 * nodes.size,
            "bkg_map_tb_s": round((8 * pix + 16 * nodes.size) / (ms['maps'] * 1e-3) / 1e12, 2),
            "snr_maps_band_ms": round(ms['engine'], 3), "engine_and_kernel_bytes_identical": same,
            "snr_finite_fraction": round(finite, 5), "file_write_s": round(write_s, 3),
            "note": "snr_kernel_ms / bkg_map_kernel_ms: CUDA events around back-to-back launches of cy_bkg_grid_snr_maps "
                    "/ cy_bkg_grid_maps into preallocated rows, the two alternating per repetition; bytes: 4 read + 8 "
                    "written per pixel (8 written for the bkg / rms maps) + 16 per node; snr_maps_band_ms: events "
                    "around Engine.snr_maps_band (row allocation, node upload, kernel); file_write_s: host clock "
                    "around both files (one rank, a temporary directory on the local disk)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='3,4')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--variant', default='l')
    ap.add_argument('--bkg_box', type=int, default=101)
    ap.add_argument('--bkg_grid', type=int, default=25)
    ap.add_argument('--mask', action='store_true', help='time the source mask (module docstring)')
    ap.add_argument('--estimator', default='mean', choices=['mean', 'median'],
                    help='median: time the median estimator against the mean (module docstring)')
    ap.add_argument('--snr', action='store_true', help='time the background-subtracted and S/N maps (module docstring)')
    ap.add_argument('--out', default=None, help='directory for bkgmap_bench.json (r05_bkgmask_bench.json with --mask, '
                                                 'r06_bkgmedian_bench.json with --estimator median, '
                                                 'r07_snrmap_bench.json with --snr)')
    a = ap.parse_args()
    info = card()
    lines = []
    for c in [int(x) for x in a.configs.split(',')]:
        fn = snr_config if a.snr else median_config if a.estimator == 'median' else mask_config if a.mask else \
            run_config
        r = fn(c, a.reps, a.variant, a.bkg_box, a.bkg_grid)
        r.update(info)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        name = 'r07_snrmap_bench.json' if a.snr else 'r06_bkgmedian_bench.json' if a.estimator == 'median' else \
            'r05_bkgmask_bench.json' if a.mask else 'bkgmap_bench.json'
        with open(os.path.join(a.out, name), 'w') as f:
            json.dump(lines, f, indent=1)


if __name__ == '__main__':
    main()
