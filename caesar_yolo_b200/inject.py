"""Catalog completeness by injection and recovery (opt-in, `inject_sources`; not part of the reference).

Beam-shaped point sources are added at empty positions of the image rows already in HBM (cy_inject_sources), the tiles
they touch are detected again, and the round's catalog is matched against the injections.  Each round starts from the
original image and records: the rows are restored word for word (cy_inject_restore) and the record slots from a
snapshot.  Definition of the beam, footprint, pixel values, S/N and placement: include/caesar_b200.h.

Everything on the host here is deterministic and identical on every rank: placement reads only the file, the
catalog (which every rank holds) and the replicated node states of the bkg / rms maps."""
import logging
import math
import time

import numpy as np
import torch

from . import ops

logger = logging.getLogger(__name__)

MAX_DRAWS = 20          # candidates drawn per requested injection and round
NBINS = 10              # log-spaced S/N bins of the completeness table
REJECT_RULES = ('outside', 'masked', 'rms', 'source', 'overlap')


def footprint_half(cov):
    """(rx, ry) = (ceil(4 sqrt(C_xx)), ceil(4 sqrt(C_yy))) of the pixel covariance of the beam."""
    return int(math.ceil(4.0 * math.sqrt(cov[0][0]))), int(math.ceil(4.0 * math.sqrt(cov[1][1])))


def inverse_cov(cov):
    """(ixx, ixy, iyy) of C_pix^-1, fp64."""
    cxx, cxy, cyy = float(cov[0][0]), float(cov[0][1]), float(cov[1][1])
    det = cxx * cyy - cxy * cxy
    return cyy / det, -cxy / det, cxx / det


def integer_boxes(src):
    """Integer boxes [ceil x1, floor x2] x [ceil y1, floor y2] of a cy_source / cy_det_record array (int64 arrays
    bx0, bx1, by0, by1; NaN coordinates give an empty box)."""
    with np.errstate(invalid='ignore'):
        c = [np.asarray(src[k], np.float64) for k in ('x1', 'x2', 'y1', 'y2')]
        bad = ~np.isfinite(c[0]) | ~np.isfinite(c[1]) | ~np.isfinite(c[2]) | ~np.isfinite(c[3])
        c = [np.where(bad, 0.0, v) for v in c]
        bx0, bx1 = np.ceil(c[0]).astype(np.int64), np.floor(c[1]).astype(np.int64)
        by0, by1 = np.ceil(c[2]).astype(np.int64), np.floor(c[3]).astype(np.int64)
    bx1[bad] = bx0[bad] - 1
    return bx0, bx1, by0, by1


def place(seed, rnd, n, region, rx, ry, boxes, centre_masked, sample_rms, snr_range):
    """Placement of round `rnd` (include/caesar_b200.h): candidates (x, y, u) = rows of
    np.random.default_rng([seed, rnd]).random((20 n, 3)), x = X0 - 1/2 + u0 W, y = R0 - 1/2 + u1 H over the region
    (X0, R0, W, H), snr = lo (hi / lo)^u2; taken in order until n are accepted.  boxes: integer_boxes of the catalog,
    in the frame of the region.  centre_masked(cx, cy) -> bool array; sample_rms(cx, cy) -> float32 array (both
    vectorised, called once for the candidates whose footprint lies in the region).
    Returns dict of arrays x, y, cx, cy, snr, rms (float32), peak (= snr * rms in fp64) of the placed injections,
    and 'drawn' and 'rejected' (count per rule of REJECT_RULES)."""
    X0, R0, W, H = region
    lo, hi = snr_range
    m = MAX_DRAWS * n
    u = np.random.default_rng([int(seed), int(rnd)]).random((m, 3))
    x = X0 - 0.5 + u[:, 0] * W
    y = R0 - 0.5 + u[:, 1] * H
    snr = lo * (hi / lo) ** u[:, 2]
    cx = np.floor(x + 0.5).astype(np.int64)
    cy = np.floor(y + 0.5).astype(np.int64)
    inside = (cx - rx >= X0) & (cx + rx <= X0 + W - 1) & (cy - ry >= R0) & (cy + ry <= R0 + H - 1)
    masked = np.zeros(m, bool)
    rms = np.full(m, np.nan, np.float32)
    k = np.flatnonzero(inside)
    if len(k):
        masked[k] = np.asarray(centre_masked(cx[k], cy[k]), bool)
        rms[k] = np.asarray(sample_rms(cx[k], cy[k]), np.float32)
    # catalog boxes dilated by the footprint, in cells of cs pixels: footprint of c meets box b <=> c in dilated b
    cs = max(128, 2 * rx + 1, 2 * ry + 1)
    cells = {}
    for b0, b1, c0, c1 in zip(*boxes):
        if b1 < b0 or c1 < c0:
            continue
        d = (int(b0) - rx, int(b1) + rx, int(c0) - ry, int(c1) + ry)
        for gy in range(d[2] // cs, d[3] // cs + 1):
            for gx in range(d[0] // cs, d[1] // cs + 1):
                cells.setdefault((gx, gy), []).append(d)
    placed = {}
    acc = []
    rej = dict.fromkeys(REJECT_RULES, 0)
    drawn = 0
    for i in range(m):
        if len(acc) == n:
            break
        drawn += 1
        if not inside[i]:
            rej['outside'] += 1
            continue
        if masked[i]:
            rej['masked'] += 1
            continue
        if not rms[i] > 0:
            rej['rms'] += 1
            continue
        px, py = int(cx[i]), int(cy[i])
        gx, gy = px // cs, py // cs
        if any(d[0] <= px <= d[1] and d[2] <= py <= d[3] for d in cells.get((gx, gy), ())):
            rej['source'] += 1
            continue
        if any(abs(px - qx) <= 2 * rx and abs(py - qy) <= 2 * ry
               for ax in (gx - 1, gx, gx + 1) for ay in (gy - 1, gy, gy + 1) for qx, qy in placed.get((ax, ay), ())):
            rej['overlap'] += 1
            continue
        placed.setdefault((gx, gy), []).append((px, py))
        acc.append(i)
    acc = np.asarray(acc, np.int64)
    out = {'x': x[acc], 'y': y[acc], 'cx': cx[acc], 'cy': cy[acc], 'snr': snr[acc], 'rms': rms[acc]}
    out['peak'] = out['snr'] * out['rms'].astype(np.float64)
    out['drawn'], out['rejected'] = drawn, rej
    return out


def affected_tiles(tiles, cx, cy, rx, ry, chunk=1024):
    """Ids of the tiles (ops.TILE_DTYPE, [xmin, xmax) x [ymin, ymax)) whose rectangle meets a footprint [cx - rx,
    cx + rx] x [cy - ry, cy + ry] (same frame as the tiles).  Only these tiles read an injected pixel."""
    hit = np.zeros(len(tiles), bool)
    tx0, tx1 = tiles['xmin'].astype(np.int64), tiles['xmax'].astype(np.int64)
    ty0, ty1 = tiles['ymin'].astype(np.int64), tiles['ymax'].astype(np.int64)
    cx, cy = np.asarray(cx, np.int64), np.asarray(cy, np.int64)
    for s in range(0, len(cx), chunk):
        a, b = cx[s:s + chunk, None], cy[s:s + chunk, None]
        hit |= ((a - rx < tx1) & (a + rx >= tx0) & (b - ry < ty1) & (b + ry >= ty0)).any(axis=0)
    return np.flatnonzero(hit).astype(np.int32)


def match(round_src, orig_src, cx, cy):
    """Injection k is recovered by the first source of round_src (catalog order) whose integer box contains (cx[k],
    cy[k]).  Returns (index of the matching source or -1 per injection, new, lost): new = round sources that are
    neither in the original catalog (same record bytes) nor matched, lost = original sources absent from the round
    catalog."""
    bx0, bx1, by0, by1 = integer_boxes(round_src)
    idx = np.full(len(cx), -1, np.int64)
    for k in range(len(cx)):
        h = np.flatnonzero((bx0 <= cx[k]) & (cx[k] <= bx1) & (by0 <= cy[k]) & (cy[k] <= by1))
        if len(h):
            idx[k] = h[0]
    orig = set(_rows(orig_src))
    rows = _rows(round_src)
    matched = set(int(i) for i in idx if i >= 0)
    new = sum(1 for i, r in enumerate(rows) if r not in orig and i not in matched)
    lost = len(orig - set(rows))
    return idx, new, lost


def _rows(src):
    a = np.ascontiguousarray(src)
    return [bytes(r) for r in a.view(np.uint8).reshape(len(a), a.dtype.itemsize)]


def snr_bin(snr, lo, hi, nbins=NBINS):
    """Bin of each S/N among nbins log-spaced bins over [lo, hi] (all in bin 0 when lo = hi)."""
    snr = np.asarray(snr, np.float64)
    if hi == lo:
        return np.zeros(len(snr), np.int64)
    return np.clip(np.floor(nbins * np.log(snr / lo) / np.log(hi / lo)).astype(np.int64), 0, nbins - 1)


def completeness(snr, recovered, lo, hi, nbins=NBINS):
    """Per S/N bin: edges, injections, recovered, fraction (None for an empty bin)."""
    edges = np.geomspace(lo, hi, nbins + 1)
    b = snr_bin(snr, lo, hi, nbins)
    rec = np.asarray(recovered, bool)
    out = []
    for i in range(nbins):
        n = int((b == i).sum())
        r = int(rec[b == i].sum())
        out.append({'snr_lo': float(edges[i]), 'snr_hi': float(edges[i + 1]), 'n': n, 'recovered': r,
                    'fraction': (r / n) if n else None})
    return out


def source_dict(s, names):
    return {'x1': float(s['x1']), 'y1': float(s['y1']), 'x2': float(s['x2']), 'y2': float(s['y2']),
            'class_id': int(s['cls']), 'class_name': str(names[int(s['cls'])]), 'score': float(s['score'])}


class Plan(object):
    """What a run hands to run_rounds.  Coordinates are in the catalog's frame.
    region: map region (X0, R0, W, H); catalog: the original catalog (ops.SRC_DTYPE, on every rank); tiles: the tile
    grid in the catalog's frame and (a, b) this rank's ids; target: (img, row_stride, big_endian, row0, ncols,
    row_begin, row_end) of the rows to inject into (None: this rank holds no rows) and x_off: buffer column of catalog
    column 0; centre_masked / sample_rms: as for place; rerun(ids): detects the tiles ids of this rank again;
    merge(): the round's catalog on rank 0 (None elsewhere)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def tiled_plan(eng, tiles, catalog, nodes, box, grid, centre_masked, rank=0, world=1):
    """The Plan of a tiled run (pipeline.run_image) on `eng`: this rank's band of rows in HBM (image columns), the map
    region of Engine.bkg_maps_band and its final node states `nodes`, the catalog and tiles in image coordinates; the
    round's catalog comes from Engine.exchange_and_merge on rank 0."""
    band, Y0, Y1, nx, big_endian = eng.band
    region = eng._map_band(tiles, rank, world)[4]
    X0, R0, W, H = region

    def sample_rms(cx, cy):
        return eng.sample_bkg_maps(nodes, W, R0, R0 + H, box, grid, np.asarray(cx) - X0, cy)[1]

    def rerun(ids):
        eng.process_tiles(band, nx, big_endian, 0, Y0, ids)
    return Plan(region=region, catalog=catalog, tiles=tiles, my_tiles=eng._my_range,
                target=None if band is None else (band, nx, big_endian, Y0, nx, Y0, Y1), x_off=0,
                centre_masked=centre_masked, sample_rms=sample_rms, rerun=rerun,
                merge=lambda: eng.exchange_and_merge(world, rank0_only=True, rank=rank)[0])


def run_rounds(eng, plan, n, rounds, snr_range, seed, cov, names, rank=0, timing=None):
    """All rounds (include/caesar_b200.h; the steps are those of README's injection section).  timing: optional dict
    that receives the summed host-clock time of each step (every step ends with a device synchronise then).
    Returns (injections, per-round records) on rank 0, None elsewhere."""
    rx, ry = footprint_half(cov)
    icov = inverse_cov(cov)
    boxes = integer_boxes(plan.catalog)
    lo, hi = snr_range
    a, b = plan.my_tiles
    snap = eng.snapshot_records()
    injections, per_round = [], []

    def step(name, t0):
        if timing is not None:
            torch.cuda.synchronize()
            timing[name] = timing.get(name, 0.0) + time.time() - t0
        return time.time()

    for r in range(rounds):
        t = time.time()
        p = place(seed, r, n, plan.region, rx, ry, boxes, plan.centre_masked, plan.sample_rms, (lo, hi))
        t = step('place_s', t)
        k = len(p['x'])
        if k < n:
            logger.warning("Injection round %d: %d of %d sources placed after %d candidates", r, k, n, p['drawn'])
        inj = np.zeros(k, ops.INJ_DTYPE)
        inj['x'], inj['y'], inj['peak'] = p['x'] + plan.x_off, p['y'], p['peak']
        inj['cx'], inj['cy'] = p['cx'] + plan.x_off, p['cy']
        handle = eng.inject(*plan.target, inj, rx, ry, icov) if plan.target is not None else None
        t = step('inject_s', t)
        ids = affected_tiles(plan.tiles, p['cx'], p['cy'], rx, ry)
        mine = ids[(ids >= a) & (ids < b)]
        plan.rerun(mine)
        t = step('rerun_s', t)
        src = plan.merge()
        t = step('merge_s', t)
        if handle is not None:
            eng.restore(handle)
        eng.restore_records(snap)
        t = step('restore_s', t)
        if timing is not None:
            timing['affected_tiles'] = timing.get('affected_tiles', 0) + len(ids)
        if rank != 0:
            continue
        idx, new, lost = match(src, plan.catalog, p['cx'], p['cy'])
        per_round.append({'round': r, 'placed': k, 'drawn': p['drawn'], 'rejected': p['rejected'],
                          'affected_tiles': int(len(ids)), 'new': int(new), 'lost': int(lost)})
        for i in range(k):
            injections.append({'round': r, 'x': float(p['x'][i]), 'y': float(p['y'][i]), 'snr': float(p['snr'][i]),
                               'rms': float(p['rms'][i]), 'peak': float(p['peak'][i]), 'recovered': bool(idx[i] >= 0),
                               'source': source_dict(src[idx[i]], names) if idx[i] >= 0 else None})
    return (injections, per_round) if rank == 0 else None


def report(image_id, injections, per_round, params):
    """The inject_<image_id>.json document."""
    lo, hi = params['snr_range']
    snr = np.array([d['snr'] for d in injections], np.float64)
    rec = np.array([d['recovered'] for d in injections], bool)
    counts = {}
    for d in injections:
        if d['recovered']:
            counts[d['source']['class_name']] = counts.get(d['source']['class_name'], 0) + 1
    return {'image_id': image_id, 'params': params, 'injections': injections,
            'completeness': completeness(snr, rec, lo, hi), 'class_counts': counts, 'rounds': per_round}
