"""Catalog reliability from the inverted image (opt-in, `reliability`; not part of the reference).

Real sources are positive, while noise and most imaging artefacts are symmetric about zero, so the detections on the
negated image -I estimate how many false detections the catalog of I holds: R = 1 - N_neg / N_pos per S/N bin.  The
rows already in HBM are negated in place (cy_negate_rows), every tile of the rank is detected again, the records are
merged into the negative catalog on every rank, the record slots are restored from a snapshot and the rows negated back
(bit for bit the original).  Both catalogs then get their peak S/N against the S/N map of the original image
(cy_source_peak_snr).  Definitions: include/caesar_b200.h, next to the injection block."""
import math
import time

import numpy as np
import torch

from . import catalog, inject

NSCORES = 10            # detection score thresholds of the score table


def score_thresholds(score_thr, n=NSCORES):
    """score_thr + k (1 - score_thr) / n, k = 0..n-1."""
    return [float(score_thr) + k * (1.0 - float(score_thr)) / n for k in range(n)]


def _ratio(n_pos, n_neg):
    return {'n_pos': int(n_pos), 'n_neg': int(n_neg), 'reliability': (1.0 - n_neg / n_pos) if n_pos else None}


def tables(snr_pos, snr_neg, score_pos, score_neg, lo, hi, score_thr):
    """The reliability tables of peak S/N arrays (NaN: no pixel) and detection scores of the catalog (pos) and the
    negative catalog (neg): per S/N bin (the bins and edges of inject.completeness over [lo, hi]), cumulative for
    S/N >= each lower edge, the counts below lo, above hi and NaN, and cumulative for score >= each threshold."""
    comp = inject.completeness([], [], lo, hi)
    edges = [d['snr_lo'] for d in comp] + [comp[-1]['snr_hi']]
    pos, neg = np.asarray(snr_pos, np.float64), np.asarray(snr_neg, np.float64)
    with np.errstate(invalid='ignore'):
        def inside(v):
            return (v >= lo) & (v <= hi)
        bp, bn = inject.snr_bin(pos[inside(pos)], lo, hi), inject.snr_bin(neg[inside(neg)], lo, hi)
        bins = [dict(snr_lo=edges[i], snr_hi=edges[i + 1], **_ratio((bp == i).sum(), (bn == i).sum()))
                for i in range(inject.NBINS)]
        cum = [dict(snr_min=edges[i], **_ratio((pos >= edges[i]).sum(), (neg >= edges[i]).sum()))
               for i in range(inject.NBINS)]
        outside = {'below': {'n_pos': int((pos < lo).sum()), 'n_neg': int((neg < lo).sum())},
                   'above': {'n_pos': int((pos > hi).sum()), 'n_neg': int((neg > hi).sum())},
                   'nan': {'n_pos': int(np.isnan(pos).sum()), 'n_neg': int(np.isnan(neg).sum())}}
    sp, sn = np.asarray(score_pos, np.float64), np.asarray(score_neg, np.float64)
    score = [dict(score_min=t, **_ratio((sp >= t).sum(), (sn >= t).sum())) for t in score_thresholds(score_thr)]
    return {'bin_edges': edges, 'snr_bins': bins, 'snr_cumulative': cum, 'snr_outside': outside, 'score_cumulative': score}


def tiled_plan(eng, tiles, catalog_src, nodes, box, grid, rank=0, world=1):
    """The inject.Plan of a tiled run (pipeline.run_image) on `eng`: this rank's band of rows in HBM and its tiles, the
    negative catalog from Engine.exchange_and_merge on every rank, and the peak S/N over this rank's rows of the map
    region of Engine.bkg_maps_band with its final node states `nodes`."""
    band, Y0, Y1, nx, big_endian = eng.band

    def rerun(ids):
        eng.process_tiles(band, nx, big_endian, 0, Y0, ids)

    def peak_snr(src, sign):
        return eng.peak_snr_band(nodes, src, tiles, box, grid, sign, rank, world)
    return inject.Plan(region=eng._map_band(tiles, rank, world)[4], catalog=catalog_src, tiles=tiles,
                       my_tiles=eng._my_range, target=None if band is None else (band, nx, big_endian, Y0, nx, Y0, Y1),
                       rerun=rerun, merge=lambda: eng.exchange_and_merge(world, rank0_only=False, rank=rank)[0],
                       peak_snr=peak_snr)


def run(eng, plan, timing=None):
    """Negative catalog and peak S/N of both catalogs (the steps of README's reliability section).  The rows and the
    record slots are left as they were.  timing: optional dict that receives the host-clock time of each step (every
    step ends with a device synchronise then).  Returns (negative catalog, (snr, x, y) of the catalog, (snr, x, y) of
    the negative catalog); every rank gets them."""
    def step(name, t0):
        if timing is not None:
            torch.cuda.synchronize()
            timing[name] = timing.get(name, 0.0) + time.time() - t0
        return time.time()

    a, b = plan.my_tiles
    t = time.time()
    snap = eng.snapshot_records()
    if plan.target is not None:
        eng.negate(*plan.target)
    t = step('negate_s', t)
    plan.rerun(np.arange(a, b, dtype=np.int32))
    t = step('rerun_s', t)
    neg = plan.merge()
    t = step('merge_s', t)
    eng.restore_records(snap)
    if plan.target is not None:     # the peak S/N reads the original rows
        eng.negate(*plan.target)
    t = step('restore_s', t)
    pos_peak = plan.peak_snr(plan.catalog, 1)
    t = step('peak_snr_catalog_s', t)
    neg_peak = plan.peak_snr(neg, -1)
    step('peak_snr_negative_s', t)
    return neg, pos_peak, neg_peak


def _num(v):
    v = float(v)
    return None if math.isnan(v) else v


def _class_counts(src, names):
    out = {}
    for c in np.asarray(src['cls'], np.int64):
        out[str(names[int(c)])] = out.get(str(names[int(c)]), 0) + 1
    return out


def negative_dicts(neg, neg_peak, names):
    """The negative detections: catalog.sources_to_dicts keys plus snr_peak and its pixel (peak_x, peak_y; null when
    no pixel of the box has an S/N)."""
    out = catalog.sources_to_dicts(neg, names)
    snr, x, y = neg_peak
    for d, s, px, py in zip(out, snr, x, y):
        d['snr_peak'] = _num(s)
        d['peak_x'], d['peak_y'] = (int(px), int(py)) if px >= 0 else (None, None)
    return out


def report(image_id, cat, neg, pos_peak, neg_peak, names, params, n_tiles_rerun):
    """The reliability_<image_id>.json document; params holds snr_range and score_thr (and the map options)."""
    lo, hi = params['snr_range']
    t = tables(pos_peak[0], neg_peak[0], cat['score'], neg['score'], lo, hi, params['score_thr'])
    params = dict(params, bin_edges=t.pop('bin_edges'), score_thresholds=score_thresholds(params['score_thr']))
    doc = {'image_id': image_id, 'params': params, 'n_catalog': int(len(cat)), 'n_negative': int(len(neg)),
           'negative_detections': negative_dicts(neg, neg_peak, names),
           'catalog_snr_peak': [_num(v) for v in pos_peak[0]]}
    doc.update(t)
    doc['class_counts'] = {'catalog': _class_counts(cat, names), 'negative': _class_counts(neg, names)}
    doc['n_tiles_rerun'] = int(n_tiles_rerun)
    return doc
