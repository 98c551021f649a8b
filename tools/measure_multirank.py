#!/usr/bin/env python
"""Per-source measurements split over ranks, under torchrun: every rank runs pipeline.run_image on its band of bench.py's
16k synthetic mosaic (config 3: YOLOv8l, full preprocessing chain), then Engine.measure_band over the rows it owns with
one all-gather of the partials, exactly as SFinder.run_parallel(measure_sources=True) does; every rank then repeats the
run alone (world 1, all rows) and compares: the catalog byte for byte, npix / peak / peak_x / peak_y exactly, the
floating-point fields within --rtol relative.  Relative differences are taken against max(|a|, |b|); `sum` is compared
against the sum of |sum| over the catalog's sources when its own value is tiny against it (a near-zero sum of signed
pixels differs by reassociation only).

usage: python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/measure_multirank.py
       (--backend gloo: the same with the ranks sharing one GPU)
With --noise, every rank also runs Engine.measure_noise_band (one all-gather of the partials per clipping pass) and
compares it with the single-rank run: nbkg, iters and the pass count exactly, bkg / rms within --rtol relative (bkg
against max(|bkg|, rms)).
With --maps, every rank also runs Engine.bkg_maps_band (the background / rms maps of the mosaic, one all-gather of the
node partials per clipping pass) and compares it with the single-rank run: node nbkg, iters and the pass count exactly,
node bkg / rms within --rtol relative (as for --noise), and its own rows of both maps within 1 float32 ulp of the same
rows of the single-rank maps (NaN positions equal).
With --mask, --noise and --maps run with the source mask of the catalog (Engine.source_mask_band, built once per run over
the rank's rows); the map comparison then also requires the same set of filled nodes (nbkg = 0 with a finite value) and
the same count of holes filled.
With --estimator median, --noise and --maps clip around the median (histograms summed with one all-reduce per digit
round); bkg, nbkg, iters and the pass count must then be identical to the single-rank run, rms within --rtol.
With --snr, every rank also runs Engine.bkg_maps_band and Engine.snr_maps_band (the background-subtracted and S/N maps of
its own rows, no collective beyond the node passes), with --mask and --estimator as given.  Its rows of both maps must be
byte-identical to the same rows of one single-rank call on the same node states (the maps do not depend on the row
split).  Against the single-rank run (its own node passes), they must be byte-identical when the node bkg / rms are; with
the mean estimator the node sums are folded in another order over 2 ranks, so the node values, and with them res / snr,
may differ in the last bits: the tool then reports the largest difference in float32 ulps (within the 1 ulp of the --maps
check, compounded by the division).

With --inject, every rank also runs --inject_rounds rounds of --inject_n source injections (inject.run_rounds, the
steps of SFinder with inject_sources, with --mask and --estimator as given) after a run over all ranks and after a
single-rank run.  The placements must be identical; with --estimator median the whole result (every injection, its
match and the per-round counts) must be; with the mean the node rms may differ in the last bits over another row split
(see --snr), so the tool reports the largest relative difference of the peaks and how many matches differ.
With --reliability, every rank also runs the reliability estimate (reliability.run, the steps of SFinder with
reliability, with --mask and --estimator as given) after a run over all ranks and after a single-rank run.  The negative
catalog must be byte for byte identical; with --estimator median the peak S/N of both catalogs must be too; with the
mean the node values may differ in the last bits over another row split (see --snr), so the tool reports the largest
relative difference of the peak S/N and how many peak pixels differ.
Prints one JSON line on rank 0 with the largest relative difference per field and the verdict of every rank."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (mosaic generator, model and thresholds of the benchmark)

FLOATS = ('sum', 'xc', 'yc', 'a', 'b', 'theta')
EXACT = ('npix', 'peak', 'peak_x', 'peak_y')


def compare(m, r):
    """Largest relative difference per float field (NaN positions must agree) and exactness of the integer fields."""
    out = {}
    for k in EXACT:
        out[k + '_exact'] = bool(np.array_equal(m[k], r[k], equal_nan=True))
    for k in FLOATS:
        a, b = m[k].astype(np.float64), r[k].astype(np.float64)
        if not np.array_equal(np.isnan(a), np.isnan(b)):
            out[k] = float('inf')
            continue
        ok = ~np.isnan(a)
        scale = np.maximum(np.abs(a[ok]), np.abs(b[ok]))
        if k == 'sum':
            scale = np.maximum(scale, 1e-6 * np.abs(b[ok]).sum())
        d = np.abs(a[ok] - b[ok]) / np.where(scale > 0, scale, 1.0)
        out[k] = float(d.max()) if d.size else 0.0
    return out


def inject_rounds(a, eng, host, tiles, rank, world):
    """--inject: source-injection rounds of the run over `world` ranks and of the single-rank run (run_image, node
    states of the maps, inject.run_rounds with --mask and --estimator).  On rank 0: the placements must be identical;
    with the median estimator the whole result must be; with the mean the node rms may differ in the last bits over
    another row split, so the largest peak difference and the injections whose match differs are reported."""
    from caesar_yolo_b200 import fits, inject, pipeline
    words = host.numpy().view(np.uint32)

    def centre_masked(cx, cy):
        v = words[cy, cx].byteswap().view(np.float32)
        return ~np.isfinite(v) | (v == 0)
    cov = fits.beam_cov_pix({"BMAJ": 0.0025, "BMIN": 0.002, "BPA": 30.0, "CDELT1": -0.0004, "CDELT2": 0.0004})
    out = []
    for r, w in ((rank, world), (0, 1)):
        src, _ = pipeline.run_image(eng, host, True, tiles, rank=r, world=w, on_rank0_only=False)
        mask = eng.source_mask_band(src, tiles, r, w) if a.mask else None
        nodes = eng.bkg_maps_band(tiles, a.bkg_box, a.bkg_grid, r, w, mask=mask, estimator=a.estimator, maps=False)[0]
        plan = inject.tiled_plan(eng, tiles, src, nodes, a.bkg_box, a.bkg_grid, centre_masked, r, w)
        out.append(inject.run_rounds(eng, plan, a.inject_n, a.inject_rounds, (3.0, 100.0), 0, cov, eng.names,
                                     rank=r))
    if rank != 0:
        return None
    (im, rm), (i1, r1) = out
    key = ('round', 'x', 'y', 'snr')
    same_place = [tuple(d[k] for k in key) for d in im] == [tuple(d[k] for k in key) for d in i1]
    identical = json.dumps([im, rm]) == json.dumps([i1, r1])
    peak = max([abs(p['peak'] - q['peak']) / max(abs(q['peak']), 1e-30) for p, q in zip(im, i1)] or [0.0])
    differ = sum(1 for p, q in zip(im, i1) if (p['recovered'], p['source']) != (q['recovered'], q['source']))
    return dict(injections=len(im), placements_identical=same_place, result_identical=identical,
                max_rel_peak_diff=peak, matches_differing=differ, rounds=rm, single_rank_rounds=r1,
                ok=bool(same_place and (a.estimator == 'mean' or identical)))


def reliability_runs(a, eng, host, tiles, rank, world):
    """--reliability: the negative catalog and the peak S/N of both catalogs of the run over `world` ranks and of the
    single-rank run (run_image, node states of the maps, reliability.run with --mask and --estimator).  On rank 0: the
    negative catalogs must be identical, and with the median estimator the peak S/N (value and pixel) too."""
    from caesar_yolo_b200 import pipeline, reliability
    out = []
    for r, w in ((rank, world), (0, 1)):
        src, _ = pipeline.run_image(eng, host, True, tiles, rank=r, world=w, on_rank0_only=False)
        mask = eng.source_mask_band(src, tiles, r, w) if a.mask else None
        nodes = eng.bkg_maps_band(tiles, a.bkg_box, a.bkg_grid, r, w, mask=mask, estimator=a.estimator, maps=False)[0]
        plan = reliability.tiled_plan(eng, tiles, src, nodes, a.bkg_box, a.bkg_grid, r, w)
        neg, pos_peak, neg_peak = reliability.run(eng, plan)
        out.append((np.array(neg, copy=True), pos_peak, neg_peak))
    if rank != 0:
        return None
    (nm, pm, qm), (n1, p1, q1) = out
    same_neg = nm.tobytes() == n1.tobytes()
    res = dict(negative_sources=int(len(n1)), negative_catalog_identical=same_neg)
    for name, m, o in (('catalog', pm, p1), ('negative', qm, q1)):
        if len(m[0]) != len(o[0]):
            res[name + '_snr_identical'] = False
            continue
        fin = np.isfinite(o[0])
        res[name + '_snr_identical'] = bool(np.array_equal(m[0].view(np.uint32), o[0].view(np.uint32)) and
                                            np.array_equal(m[1], o[1]) and np.array_equal(m[2], o[2]))
        d = np.abs(m[0][fin].astype(np.float64) - o[0][fin]) / np.maximum(np.abs(o[0][fin]), 1e-30)
        res[name + '_max_rel_snr_diff'] = float(d.max()) if len(d) else 0.0
        res[name + '_peak_pixels_differing'] = int(((m[1] != o[1]) | (m[2] != o[2])).sum())
    res['ok'] = bool(same_neg and (a.estimator == 'mean' or (res.get('catalog_snr_identical') and
                                                            res.get('negative_snr_identical'))))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--mosaic', type=int, default=16384)
    ap.add_argument('--variant', default='l')
    ap.add_argument('--rtol', type=float, default=1e-12)
    ap.add_argument('--backend', default='nccl', choices=['nccl', 'gloo'],
                    help='gloo lets several ranks share one GPU (NCCL needs one GPU per rank)')
    ap.add_argument('--noise', action='store_true', help='also compare the local background / noise')
    ap.add_argument('--noise_frame', type=int, default=16)
    ap.add_argument('--maps', action='store_true', help='also compare the background / rms maps')
    ap.add_argument('--bkg_box', type=int, default=101)
    ap.add_argument('--bkg_grid', type=int, default=25)
    ap.add_argument('--mask', action='store_true', help='run --noise and --maps with the source mask')
    ap.add_argument('--estimator', default='mean', choices=['mean', 'median'],
                    help='centre of the --noise, --maps and --snr clipping')
    ap.add_argument('--snr', action='store_true', help='also compare the background-subtracted and S/N maps')
    ap.add_argument('--inject', action='store_true', help='also compare source-injection rounds')
    ap.add_argument('--inject_n', type=int, default=1024)
    ap.add_argument('--inject_rounds', type=int, default=2)
    ap.add_argument('--reliability', action='store_true', help='also compare the reliability estimate')
    a = ap.parse_args()
    import torch
    import torch.distributed as dist
    from caesar_yolo_b200 import ops, pipeline, weights as W
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    local %= torch.cuda.device_count()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if a.backend == 'nccl':
        dist.init_process_group('nccl', device_id=dev)
    else:
        dist.init_process_group('gloo')
    _, host = bench.make_mosaic_pinned(argparse.Namespace(mosaic=a.mosaic))
    n = a.mosaic
    tiles = ops.generate_tiles(0, n - 1, 0, n - 1, 512, 512, 1.0, 1.0)
    w = W.make_random_weights(a.variant, 5, seed=0, cls_bias=bench.CLS_BIAS.get(a.variant, -16.0))
    eng = pipeline.Engine(w, pipeline.make_pp_config(**bench.PP_FLAGS), imgsz=640, score_thr=bench.SCORE_THR,
                          iou_thr=bench.IOU_THR, thr_soft=bench.SOFT, thr_hard=bench.HARD, device=dev)
    src, _ = pipeline.run_image(eng, host, True, tiles, rank=rank, world=world, on_rank0_only=False)
    meas = eng.measure_band(src, tiles, rank, world)
    rows = pipeline.measure_rows(tiles, world)[rank]
    ref, _ = pipeline.run_image(eng, host, True, tiles)
    ref_meas = eng.measure_band(ref, tiles)
    res = compare(meas, ref_meas)
    same_catalog = bool(src.tobytes() == ref.tobytes())
    ok = same_catalog and all(res[k + '_exact'] for k in EXACT) and all(res[k] <= a.rtol for k in FLOATS)
    mask = eng.source_mask_band(src, tiles, rank, world) if a.mask else None
    ref_mask = eng.source_mask_band(ref, tiles) if a.mask else None
    noise_res = None
    if a.noise:
        z = eng.measure_noise_band(src, tiles, a.noise_frame, rank, world, mask=mask, estimator=a.estimator)
        passes = eng.noise_passes
        zr = eng.measure_noise_band(ref, tiles, a.noise_frame, mask=ref_mask, estimator=a.estimator)
        noise_res = dict(passes=passes, single_rank_passes=eng.noise_passes,
                         nbkg_exact=bool(np.array_equal(z['nbkg'], zr['nbkg'])),
                         iters_exact=bool(np.array_equal(z['iters'], zr['iters'])))
        for k in ('bkg', 'rms'):
            x, y = z[k], zr[k]
            same_nan = np.array_equal(np.isnan(x), np.isnan(y))
            f = ~np.isnan(y)
            scale = np.maximum(np.abs(x[f]), np.abs(y[f]))
            if k == 'bkg':   # a mean near 0 is compared at the scale of the frame's spread
                scale = np.maximum(scale, zr['rms'][f])
            dd = np.abs(x[f] - y[f]) / np.where(scale > 0, scale, 1.0)
            noise_res[k] = float(dd.max()) if (same_nan and dd.size) else (0.0 if same_nan else float('inf'))
        noise_res['bkg_identical'] = bool(np.array_equal(z['bkg'], zr['bkg'], equal_nan=True))
        ok = ok and noise_res['nbkg_exact'] and noise_res['iters_exact'] and passes == eng.noise_passes and \
            noise_res['bkg'] <= a.rtol and noise_res['rms'] <= a.rtol and \
            (a.estimator == 'mean' or noise_res['bkg_identical'])
    maps_res = None
    if a.maps:
        z, bkg, rms, _, (r0, r1) = eng.bkg_maps_band(tiles, a.bkg_box, a.bkg_grid, rank, world, mask=mask,
                                                     estimator=a.estimator)
        passes, filled = eng.bkg_passes, eng.bkg_holes_filled
        zr, bkg_r, rms_r, _, _ = eng.bkg_maps_band(tiles, a.bkg_box, a.bkg_grid, mask=ref_mask, estimator=a.estimator)
        maps_res = dict(passes=passes, single_rank_passes=eng.bkg_passes, nodes=int(z.size),
                        nbkg_exact=bool(np.array_equal(z['nbkg'], zr['nbkg'])),
                        iters_exact=bool(np.array_equal(z['iters'], zr['iters'])))
        if a.mask:
            maps_res.update(holes_filled=filled, single_rank_holes_filled=eng.bkg_holes_filled,
                            filled_set_exact=bool(np.array_equal((z['nbkg'] == 0) & ~np.isnan(z['bkg']),
                                                                 (zr['nbkg'] == 0) & ~np.isnan(zr['bkg']))))
            ok = ok and maps_res['filled_set_exact'] and filled == eng.bkg_holes_filled
        for k in ('bkg', 'rms'):
            x, y = z[k].ravel(), zr[k].ravel()
            same_nan = np.array_equal(np.isnan(x), np.isnan(y))
            f = ~np.isnan(y)
            scale = np.maximum(np.abs(x[f]), np.abs(y[f]))
            if k == 'bkg':
                scale = np.maximum(scale, zr['rms'].ravel()[f])
            dd = np.abs(x[f] - y[f]) / np.where(scale > 0, scale, 1.0)
            maps_res[k] = float(dd.max()) if (same_nan and dd.size) else (0.0 if same_nan else float('inf'))
        ulp = 0.0
        for mine, ref in ((bkg, bkg_r), (rms, rms_r)):
            p = mine.cpu().numpy().view('>f4').astype(np.float64)
            q = ref[r0 - tiles['ymin'].min():r1 - tiles['ymin'].min()].cpu().numpy().view('>f4').astype(np.float32)
            if not np.array_equal(np.isnan(p), np.isnan(q)):
                ulp = float('inf')
                break
            f = ~np.isnan(q)
            if f.any():
                ulp = max(ulp, float((np.abs(p[f] - q[f]) / np.spacing(np.abs(q[f]))).max()))
        maps_res['map_max_ulp'] = ulp
        maps_res['bkg_identical'] = bool(np.array_equal(z['bkg'], zr['bkg'], equal_nan=True))
        ok = ok and maps_res['nbkg_exact'] and maps_res['iters_exact'] and passes == eng.bkg_passes and \
            maps_res['bkg'] <= a.rtol and maps_res['rms'] <= a.rtol and ulp <= 1.0 and \
            (a.estimator == 'mean' or maps_res['bkg_identical'])
    snr_res = None
    if a.snr:
        z = eng.bkg_maps_band(tiles, a.bkg_box, a.bkg_grid, rank, world, mask=mask, estimator=a.estimator)[0]
        res_m, snr_m, _, (r0, r1) = eng.snr_maps_band(z, tiles, a.bkg_box, a.bkg_grid, rank, world)
        zr = eng.bkg_maps_band(tiles, a.bkg_box, a.bkg_grid, mask=ref_mask, estimator=a.estimator)[0]
        y0 = int(tiles['ymin'].min())
        res_s, snr_s, _, _ = eng.snr_maps_band(z, tiles, a.bkg_box, a.bkg_grid)   # the same nodes, all rows at once
        split_ok = bool(torch.equal(res_m, res_s[r0 - y0:r1 - y0]) and torch.equal(snr_m, snr_s[r0 - y0:r1 - y0]))
        res_r, snr_r, _, _ = eng.snr_maps_band(zr, tiles, a.bkg_box, a.bkg_grid)
        same_nodes = all(z[k].tobytes() == zr[k].tobytes() for k in ('bkg', 'rms'))
        snr_res = dict(rows=[r0, r1], row_split_identical=split_ok, node_bkg_rms_identical=same_nodes,
                       res_identical=bool(torch.equal(res_m, res_r[r0 - y0:r1 - y0])),
                       snr_identical=bool(torch.equal(snr_m, snr_r[r0 - y0:r1 - y0])))
        for k, mine, ref_rows in (('res', res_m, res_r), ('snr', snr_m, snr_r)):
            p = mine.cpu().numpy().view('>f4').astype(np.float64)
            q = ref_rows[r0 - y0:r1 - y0].cpu().numpy().view('>f4').astype(np.float32)
            f = ~np.isnan(q)
            same_nan = np.array_equal(np.isnan(p), ~f)
            ulp = float((np.abs(p[f] - q[f]) / np.spacing(np.abs(q[f]))).max()) if f.any() else 0.0
            snr_res[k + '_max_ulp'] = ulp if same_nan else float('inf')
        ok = ok and split_ok and (not same_nodes or (snr_res['res_identical'] and snr_res['snr_identical']))
    inject_res = None
    if a.inject:
        inject_res = inject_rounds(a, eng, host, tiles, rank, world)
        ok = ok and (rank != 0 or inject_res['ok'])
    rel_res = None
    if a.reliability:
        rel_res = reliability_runs(a, eng, host, tiles, rank, world)
        ok = ok and (rank != 0 or rel_res['ok'])
    flags = torch.tensor([1 if ok else 0], device=dev if a.backend == 'nccl' else 'cpu')
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(json.dumps(dict(world=world, backend=a.backend, gpus=torch.cuda.device_count(), mosaic=n,
                              sources=int(len(src)), rows_of_rank0=list(rows),
                              catalog_identical=same_catalog, max_rel_diff={k: res[k] for k in FLOATS},
                              exact={k: res[k + '_exact'] for k in EXACT}, rtol=a.rtol, estimator=a.estimator,
                              noise=noise_res, maps=maps_res, snr=snr_res, inject=inject_res,
                              reliability=rel_res,
                              matches_single_rank_on_every_rank=bool(int(flags[0])))), flush=True)
    dist.destroy_process_group()
    return 0 if int(flags[0]) else 1


if __name__ == '__main__':
    sys.exit(main())
