"""Catalog / region writers with the reference's file formats (SURVEY App. C): `catalog_<image_id>.json`
(SFinder.write_json_results, caesar_yolo/inference.py:1196-1211), `out_<image_id>.json`
(Analyzer.write_json_results, caesar_yolo/evaluation.py:472-483) and the DS9 region text the `regions` package emits
(inference.py:1214-1287, evaluation.py:487-548; `regions` itself is not a dependency)."""
import json
import math

CLASS_COLOR_DS9 = {  # SFinder (mosaic catalog), inference.py:334-342
    'bkg': "black", 'spurious': "red", 'compact': "blue", 'extended': "green", 'extended-multisland': "yellow",
    'flagged': "black", 'diffuse': "magenta",
}
CLASS_COLOR_DS9_ANALYZER = {  # Analyzer (single image / per-tile files), evaluation.py:108-115
    'bkg': "black", 'spurious': "red", 'compact': "blue", 'extended': "green", 'extended-multisland': "orange",
    'flagged': "magenta",
}


# per-source measurement keys (Engine.measure + fits metadata); written only when measurements are requested
MEASURE_KEYS = ('npix', 'sum', 'peak', 'peak_x', 'peak_y', 'xc', 'yc', 'a', 'b', 'theta', 'flux', 'ra', 'dec')


def _num(v):
    v = float(v)
    return v if math.isfinite(v) else None      # JSON null


# local background / noise keys (Engine.measure_noise); written only when the noise is measured
NOISE_KEYS = ('bkg', 'rms', 'nbkg', 'snr', 'flux_bkgsub', 'flux_err')


def measurement_dicts(meas, beam_area_pix=None, radec=None, noise=None):
    """ops.MEAS_DTYPE array -> one dict of MEASURE_KEYS per source.  flux = sum / beam_area_pix (None without a beam);
    radec: (ra, dec) arrays of the centroids in degrees, or None.  noise: ops.NOISE_DTYPE array of the same sources, or
    None; with it the dicts also get NOISE_KEYS (noise_keys).  Non-finite values become None (JSON null)."""
    out = []
    for i, m in enumerate(meas):
        d = {"npix": int(m['npix'])}
        for k in MEASURE_KEYS[1:10]:
            d[k] = _num(m[k])
        d["flux"] = _num(m['sum'] / beam_area_pix) if beam_area_pix else None
        d["ra"] = _num(radec[0][i]) if radec is not None else None
        d["dec"] = _num(radec[1][i]) if radec is not None else None
        if noise is not None:
            d.update(noise_keys(m, noise[i], beam_area_pix))
        out.append(d)
    return out


def noise_keys(m, z, beam_area_pix=None):
    """NOISE_KEYS of one source from its measurements m (ops.MEAS_DTYPE) and clipped frame statistics z
    (ops.NOISE_DTYPE), A = beam_area_pix:
      bkg, rms     clipped mean / std of the frame (None when nbkg = 0)
      nbkg         pixels in the final kept set
      snr          (peak - bkg) / rms (None without a peak, when nbkg = 0 or rms = 0)
      flux_bkgsub  (sum - npix * bkg) / A
      flux_err     rms * sqrt(npix * min(npix, A)) / A: the noise taken as correlated over one beam, so it is
                   rms * sqrt(npix / A) for a box much larger than the beam and rms * npix / A for one smaller than it
    (flux_bkgsub and flux_err are None without a beam area or when nbkg = 0)."""
    nb = int(z['nbkg'])
    d = {"nbkg": nb, "bkg": None, "rms": None, "snr": None, "flux_bkgsub": None, "flux_err": None}
    if nb == 0:
        return d
    bkg, rms, npix = float(z['bkg']), float(z['rms']), int(m['npix'])
    d["bkg"], d["rms"] = _num(bkg), _num(rms)
    if npix > 0 and rms > 0:
        d["snr"] = _num((float(m['peak']) - bkg) / rms)
    if beam_area_pix:
        A = float(beam_area_pix)
        d["flux_bkgsub"] = _num((float(m['sum']) - npix * bkg) / A)
        d["flux_err"] = _num(rms * math.sqrt(npix * min(npix, A)) / A)
    return d


def sources_to_dicts(src, names, meas=None):
    """cy_source array -> list of dicts with the reference's keys.  Pass-through sources keep the reference's mixed
    `edge` typing (int 0 from make_json_results, True once find_sources_at_edge fired).  meas: optional
    measurement_dicts of the same sources, whose keys are added."""
    out = []
    for i, s in enumerate(src):
        edge = bool(int(s['flags']) & 1)
        out.append({
            "name": "S%d" % (i + 1),
            "x1": float(s['x1']), "x2": float(s['x2']), "y1": float(s['y1']), "y2": float(s['y2']),
            "class_id": int(s['cls']), "class_name": str(names[int(s['cls'])]), "score": float(s['score']),
            "edge": True if edge else 0, "merged": bool(int(s['flags']) & 2),
        })
        if meas is not None:
            out[-1].update(meas[i])
    return out


def records_to_objs(recs, names, tag="", meas=None):
    """cy_det_record array of ONE image/tile -> Analyzer.results['objs'] (evaluation.py:418-469).  meas: optional
    measurement_dicts of the same records, whose keys are added."""
    objs = []
    for i, r in enumerate(recs):
        name = 'S' + str(i + 1) if tag == "" else 'S' + str(i + 1) + "_" + tag
        objs.append({"name": name, "x1": float(r['x1']), "x2": float(r['x2']), "y1": float(r['y1']),
                     "y2": float(r['y2']), "class_id": int(r['cls']), "class_name": str(names[int(r['cls'])]),
                     "score": float(r['score']), "edge": int(int(r['flags']) & 1)})
        if meas is not None:
            objs[-1].update(meas[i])
    return objs


def write_json(obj, path):
    with open(path, 'w') as fp:
        json.dump(obj, fp, indent=2, sort_keys=True)


def _fmt(v):
    return ("%.4f" % v).rstrip('0').rstrip('.') if v != int(v) else "%d" % int(v)


def write_ds9(dicts, path, merged_key=True):
    """One `box` per source: centre (x1 + dx/2, y1 + dy/2) in 1-based image coordinates, text/tag/color metadata.
    merged_key=True: SFinder.make_ds9_regions (inference.py:1214-1263, its colour map, MERGED tag);
    False: Analyzer.make_ds9_regions (evaluation.py:487-528).  Like the reference, nothing is written for an empty
    list and an unknown class name raises KeyError."""
    if not dicts:
        return
    colors = CLASS_COLOR_DS9 if merged_key else CLASS_COLOR_DS9_ANALYZER
    lines = ["# Region file format: DS9 astropy/regions", "image"]
    for d in dicts:
        dx, dy = d['x2'] - d['x1'], d['y2'] - d['y1']
        xc, yc = d['x1'] + 0.5 * dx, d['y1'] + 0.5 * dy
        tags = [d['class_name']]
        if d.get('edge'):
            tags.append('BORDER')
        if merged_key and d.get('merged'):
            tags.append('MERGED')
        meta = "text={%s} " % d['name'] + " ".join("tag={%s}" % t for t in tags)
        lines.append("box(%s,%s,%s,%s,0) # %s color=%s" % (_fmt(xc + 1), _fmt(yc + 1), _fmt(dx), _fmt(dy), meta,
                                                            colors[d['class_name']]))
    with open(path, 'w') as fp:
        fp.write("\n".join(lines) + "\n")


def write_tile_outputs(recs, tiles, tile_ids, status, names, image_id, outdir, save_json, save_regions):
    """Per-tile files of TileTask.find_sources (inference.py:218-229): `catalog_<id>_tid<N>.json` /
    `catalog_<id>_tid<N>.reg`, written by Analyzer.predict (evaluation.py:216-234) for every tile whose prediction
    ran (rejected tiles return before writing), with tile-local `edge` flags and names `S<k>_t<N>`.
    recs: cy_det_record array of this rank (tile-id order); status[i] < 0: tile tile_ids[i] was rejected."""
    import os
    import numpy as np
    order = np.argsort(recs['tile_id'], kind='stable')
    recs = recs[order]
    bounds = np.searchsorted(recs['tile_id'], np.asarray(tile_ids), side='left')
    bounds_hi = np.searchsorted(recs['tile_id'], np.asarray(tile_ids), side='right')
    written = []
    for k, tid in enumerate(tile_ids):
        if status is not None and status[k] < 0:
            continue
        objs = records_to_objs(recs[bounds[k]:bounds_hi[k]], names, tag="t" + str(int(tid)))
        base = os.path.join(outdir, 'catalog_' + str(image_id) + '_tid' + str(int(tid)))
        if save_json:
            write_json({"image_id": image_id, "objs": objs}, base + '.json')
            written.append(base + '.json')
        if save_regions and objs:
            write_ds9(objs, base + '.reg', merged_key=False)
            written.append(base + '.reg')
    return written
