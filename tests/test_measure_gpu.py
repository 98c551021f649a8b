"""Per-source measurements on the GPU (cy_measure_sources / cy_measure_combine, Engine.measure, SFinder with
measure_sources=True) against a numpy fp64 restatement of the same definitions.

Tolerances: npix, peak, peak_x, peak_y are exact.  The sums are compared relative to the sum of the absolute values of
their terms (the scale at which a reordered fp64 sum can differ), at 1e-12; the values derived from them as _close_derived
states."""
import json
import math

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import ops, synth

pytestmark = pytest.mark.gpu

SUMS = ('sum', 'sw', 'swx', 'swy', 'swxx', 'swyy', 'swxy')


def ref_measure(img, boxes, r0=0, r1=None):
    """numpy restatement.  img: 2-D float32 (decoded values, NaN allowed); boxes [n, 4] = x1, y1, x2, y2 inclusive.
    Returns (partial sums dict of arrays, abs-scale dict of arrays, final values dict of arrays)."""
    ny, nx = img.shape
    r1 = ny if r1 is None else r1
    n = len(boxes)
    P = {k: np.zeros(n) for k in SUMS}
    S = {k: np.zeros(n) for k in SUMS}
    M = {k: np.full(n, np.nan) for k in ('peak', 'peak_x', 'peak_y', 'xc', 'yc', 'a', 'b', 'theta')}
    M['npix'] = np.zeros(n, np.int64)
    for i, (x1, y1, x2, y2) in enumerate(np.asarray(boxes, np.float64)):
        cx, cy = math.ceil(x1), math.ceil(y1)
        xa, xb = max(math.ceil(x1), 0), min(math.floor(x2), nx - 1)
        ya, yb = max(math.ceil(y1), r0), min(math.floor(y2), r1 - 1)
        if xa > xb or ya > yb:
            continue
        sub = img[ya:yb + 1, xa:xb + 1].astype(np.float64)
        with np.errstate(invalid='ignore'):
            m = np.isfinite(sub) & (sub != 0)
        yy, xx = np.nonzero(m)
        v = sub[m]
        M['npix'][i] = v.size
        if v.size == 0:
            continue
        k = int(np.argmax(v))                      # first maximum in row-major order = lowest index
        M['peak'][i], M['peak_x'][i], M['peak_y'][i] = v[k], xx[k] + xa, yy[k] + ya
        w = np.maximum(v, 0.0)
        dx = (xx + xa - cx).astype(np.float64)
        dy = (yy + ya - cy).astype(np.float64)
        terms = dict(sum=v, sw=w, swx=w * dx, swy=w * dy, swxx=w * dx * dx, swyy=w * dy * dy, swxy=w * dx * dy)
        for key, t in terms.items():
            P[key][i] = t.sum()
            S[key][i] = np.abs(t).sum()
        sw = P['sw'][i]
        if sw > 0:
            mx, my = P['swx'][i] / sw, P['swy'][i] / sw
            M['xc'][i], M['yc'][i] = mx + cx, my + cy
            cxx = max(P['swxx'][i] / sw - mx * mx, 0.0)
            cyy = max(P['swyy'][i] / sw - my * my, 0.0)
            cxy = P['swxy'][i] / sw - mx * my
            h, d = 0.5 * (cxx + cyy), math.sqrt(0.25 * (cxx - cyy) ** 2 + cxy * cxy)
            M['a'][i], M['b'][i] = math.sqrt(h + d), math.sqrt(max(h - d, 0.0))
            th = math.degrees(0.5 * math.atan2(2 * cxy, cxx - cyy))
            M['theta'][i] = th + 180.0 if th <= -90.0 else th
    M['sum'] = P['sum']
    return P, S, M


def _src(boxes):
    s = np.zeros(len(boxes), dtype=ops.SRC_DTYPE)
    b = np.asarray(boxes, np.float32)
    s['x1'], s['y1'], s['x2'], s['y2'] = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    return s


def _gpu(img_words, big_endian, ncols, boxes, ranges, dev, row0s=None):
    """Measure over each row range (separate calls, each on a buffer starting at its own first row when row0s is given),
    then combine in range order.  -> (partials [len(ranges), n] PARTIAL_DTYPE, meas MEAS_DTYPE)."""
    src = _src(boxes)
    src_dev = ops.to_device_bytes(src, dev)
    n = len(src)
    parts = []
    full = torch.from_numpy(np.ascontiguousarray(img_words)).to(dev)
    for k, (r0, r1) in enumerate(ranges):
        if row0s is not None:
            buf, row0 = full[r0:max(r1, r0 + 1)], r0
        else:
            buf, row0 = full, 0
        parts.append(ops.measure_sources(buf, ncols, big_endian, row0, ncols, src_dev, n, r0, r1).clone())
    allp = torch.cat(parts)
    meas = ops.measure_combine(allp, len(ranges), src_dev, n, ncols)
    torch.cuda.synchronize()
    return (allp.cpu().numpy().view(ops.PARTIAL_DTYPE).reshape(len(ranges), n),
            meas.cpu().numpy().view(ops.MEAS_DTYPE))


def _moment_scale(P):
    """Mean squared offset of the weight from the box corner, (sum w*dx^2 + sum w*dy^2) / sum w, per source.  The central
    second moments are that raw moment minus the squared centroid offset, so their rounding error scales with it."""
    with np.errstate(invalid='ignore', divide='ignore'):
        return (P['swxx'] + P['swyy']) / P['sw']


def _close_derived(g, r, q):
    """Centroid at 1e-9 relative.  a and b: their squares (the eigenvalues of the central second-moment matrix) within
    1e-9 relative plus 1e-11 of the raw moment scale q (_moment_scale) — the cancellation the central moments carry,
    which only matters where a true moment is about 0 (one-pixel or one-row weight); theta where it is well defined
    (a > 0.5 px, a - b > 1 % of a)."""
    for k in ('xc', 'yc'):
        np.testing.assert_allclose(g[k], r[k], rtol=1e-9, atol=1e-9, equal_nan=True, err_msg=k)
    for k in ('a', 'b'):
        gk, rk = np.asarray(g[k], np.float64), np.asarray(r[k], np.float64)
        np.testing.assert_array_equal(np.isnan(gk), np.isnan(rk), err_msg=k)
        ok = ~np.isnan(rk)
        err = np.abs(gk[ok] ** 2 - rk[ok] ** 2)
        assert np.all(err <= 1e-9 * rk[ok] ** 2 + 1e-11 * q[ok]), (k, float((err / (rk[ok] ** 2 + q[ok])).max()))
    a, b = np.asarray(r['a'], np.float64), np.asarray(r['b'], np.float64)
    gt, rt = np.asarray(g['theta'], np.float64), np.asarray(r['theta'], np.float64)
    np.testing.assert_array_equal(np.isnan(gt), np.isnan(rt))
    with np.errstate(invalid='ignore'):
        ok = np.isfinite(a) & (a > 0.5) & (a - b > 0.01 * a)
    assert np.all(np.abs((gt[ok] - rt[ok] + 90.0) % 180.0 - 90.0) < 1e-5)
    assert np.all((gt[~np.isnan(gt)] > -90.0) & (gt[~np.isnan(gt)] <= 90.0))


def _check(meas, P, S, M, part=None):
    np.testing.assert_array_equal(meas['npix'], M['npix'])
    for k in ('peak', 'peak_x', 'peak_y'):
        np.testing.assert_array_equal(meas[k], M[k], err_msg=k)
    assert np.all(np.abs(meas['sum'] - P['sum']) <= 1e-12 * S['sum'])
    if part is not None:   # one range: the partial sums themselves
        for k in SUMS:
            assert np.all(np.abs(part[k] - P[k]) <= 1e-12 * S[k]), k
    _close_derived(meas, M, _moment_scale(P))


def _test_mosaic(seed):
    """Synthetic mosaic (NaN border) with a zero block, a negative-only block and a block of tied maxima."""
    img = synth.make_mosaic(2300, 2200, seed=seed, nan_border_frac=0.02)
    img[300:340, 500:560] = 0.0
    img[400:430, 700:740] = -np.abs(img[400:430, 700:740]) - 1e-4
    img[600:620, 900:930] = 1e-4
    img[605, 910] = img[612, 905] = img[612, 925] = 0.5                 # three tied peaks
    img[700:704, 1000:1040] = np.nan                                      # a NaN block inside a box
    return img


def _boxes(img, seed):
    ny, nx = img.shape
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(-20, nx + 20, 300), rng.uniform(-20, ny + 20, 300)
    w, h = np.exp(rng.uniform(0, np.log(80), 300)), np.exp(rng.uniform(0, np.log(80), 300))
    b = np.floor(np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1))
    special = [
        (-15, -10, 30, 40), (nx - 20, ny - 8, nx + 30, ny + 5), (nx - 1, 50, nx + 10, 60),   # clipped by the edges
        (100, 200, 100, 200), (1234, 777, 1234, 777),                                          # 1 x 1
        (300, 1000, 420, 1000), (0, 1500, nx - 1, 1500),                                       # 1 row
        (10, 10, 30, 30), (0, 0, nx - 1, 20),                                                  # all NaN (border)
        (505, 305, 550, 335),                                                                  # all zero
        (702, 402, 735, 428),                                                                  # negative only
        (900, 600, 929, 619), (899, 599, 930, 620),                                            # tied peaks
        (995, 690, 1045, 710),                                                                 # NaN block inside
        (80, 120, 2180, 2250),                                                                 # hull > 2000 x 2000
        (5000, 10, 5010, 20), (10, 5000, 20, 5010), (50, 60, 40, 70),                          # empty
    ]
    return np.concatenate([b, np.asarray(special, np.float64)])


@pytest.mark.parametrize("big_endian", [True, False])
def test_parity_with_numpy(cuda_dev, big_endian):
    img = _test_mosaic(5)
    boxes = _boxes(img, 6)
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    part, meas = _gpu(words, big_endian, img.shape[1], boxes, [(0, img.shape[0])], cuda_dev)
    P, S, M = ref_measure(img, boxes)
    _check(meas, P, S, M, part[0])
    # the special cases do what they say
    k0 = len(boxes) - 18
    assert meas['npix'][k0 + 7] == 0 and np.isnan(meas['xc'][k0 + 7]) and np.isnan(meas['peak'][k0 + 7])
    assert meas['npix'][k0 + 9] == 0 and np.isnan(meas['xc'][k0 + 9])
    assert meas['npix'][k0 + 10] > 0 and meas['peak'][k0 + 10] < 0 and np.isnan(meas['xc'][k0 + 10])
    assert (meas['peak_x'][k0 + 11], meas['peak_y'][k0 + 11]) == (910, 605)
    assert meas['npix'][k0 + 14] > 4_000_000
    assert np.all(meas['npix'][-3:] == 0)


def test_row_split_invariance(cuda_dev):
    img = _test_mosaic(7)
    boxes = _boxes(img, 8)
    ny, nx = img.shape
    words = img.astype('>f4').view(np.int32)
    _, one = _gpu(words, True, nx, boxes, [(0, ny)], cuda_dev)
    P, S, _ = ref_measure(img, boxes)
    # boundaries through the middle of boxes (the hull, the tie box, random ones), an empty range, uneven widths
    for cuts in ([610], [333, 1111, 1500], [1, 2, 3, 1000, 1000, 2299], list(range(97, ny, 97))):
        edges = [0] + cuts + [ny]
        ranges = list(zip(edges[:-1], edges[1:]))
        _, got = _gpu(words, True, nx, boxes, ranges, cuda_dev, row0s=True)
        for k in ('npix', 'peak', 'peak_x', 'peak_y'):
            np.testing.assert_array_equal(got[k], one[k], err_msg=k)
        assert np.all(np.abs(got['sum'] - one['sum']) <= 1e-12 * S['sum'])
        _close_derived(got, one, _moment_scale(P))


def test_physics_gaussians(cuda_dev):
    """Isolated elliptical Gaussians on a noiseless image: centroid, integral and shape recovered."""
    ny, nx = 600, 900
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float64)
    cases = [  # x0, y0, amplitude, sigma_major, sigma_minor, theta (deg, from +x towards +y)
        (150.3, 140.7, 2.0, 6.0, 3.0, 30.0), (450.0, 150.5, 0.01, 4.0, 4.0 * 0.6, -60.0),
        (750.6, 160.2, 5.0, 8.0, 2.5, 90.0), (200.2, 440.4, 1.0, 3.0, 1.8, 0.0), (600.7, 430.1, 0.3, 10.0, 5.0, 75.0)]
    img = np.zeros((ny, nx))
    boxes = []
    for x0, y0, A, sa, sb, th in cases:
        t = math.radians(th)
        u = math.cos(t) * (xx - x0) + math.sin(t) * (yy - y0)
        v = -math.sin(t) * (xx - x0) + math.cos(t) * (yy - y0)
        img += A * np.exp(-0.5 * ((u / sa) ** 2 + (v / sb) ** 2))
        r = 7 * sa
        boxes.append((math.floor(x0 - r), math.floor(y0 - r), math.ceil(x0 + r), math.ceil(y0 + r)))
    img = img.astype(np.float32)
    img[img < 1e-30] = 0
    _, meas = _gpu(img.view(np.int32), False, nx, boxes, [(0, ny)], cuda_dev)
    beam_area = 17.3   # any beam: flux * beam_area is the integral
    for m, (x0, y0, A, sa, sb, th) in zip(meas, cases):
        assert abs(m['xc'] - x0) < 0.05 and abs(m['yc'] - y0) < 0.05
        flux = m['sum'] / beam_area
        assert abs(flux * beam_area / (2 * math.pi * A * sa * sb) - 1) < 0.01
        assert abs(m['a'] / sa - 1) < 0.02 and abs(m['b'] / sb - 1) < 0.02
        dth = (m['theta'] - th + 90.0) % 180.0 - 90.0
        if sa != sb:
            assert abs(dth) <= 0.02 * max(abs(th), 45.0), (m['theta'], th)


# ---------------------------------------------------------------------------------------------- end to end

WCS_CARDS = {"BMAJ": 0.0025, "BMIN": 0.002, "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN", "CRVAL1": 150.0,
             "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.0, "CDELT1": -0.0004, "CDELT2": 0.0004}
MKEYS = ('npix', 'sum', 'peak', 'peak_x', 'peak_y', 'xc', 'yc', 'a', 'b', 'theta', 'flux', 'ra', 'dec')


def _config(path, outdir, split, **kw):
    cfg = dict(img_size=640, preprocess_fcn=None, image_path=path, image_xmin=-1, image_xmax=-1, image_ymin=-1,
               image_ymax=-1, mpi=None, split_image_in_tiles=split, tile_xsize=512, tile_ysize=512, tile_xstep=1.0,
               tile_ystep=1.0, max_ntasks_per_worker=10000, devices=['cuda:0'], use_multi_gpu=False, iou_thr=0.5,
               merge_overlap_iou_thr_soft=0.3, merge_overlap_iou_thr_hard=0.8, score_thr=0.5, save_catalog=True,
               save_region=True, outdir=outdir)
    cfg.update(kw)
    return cfg


def _pp(full):
    from caesar_yolo_b200.preprocessing import (BkgSubtractor, SigmaClipper, ChanResizer, ZScaleTransformer,
                                                Chan3Trasformer, MinMaxNormalizer, DataPreprocessor)
    if not full:
        return DataPreprocessor([ZScaleTransformer(contrasts=[.25, .25, .25]), MinMaxNormalizer(norm_min=0, norm_max=255.)])
    return DataPreprocessor([BkgSubtractor(sigma=3), SigmaClipper(sigma_low=10, sigma_up=10), ChanResizer(nchans=3),
                             ZScaleTransformer(contrasts=[.25, .25, .25]),
                             Chan3Trasformer(sigma_clip_baseline=0, sigma_clip_low=10, sigma_clip_up=10,
                                             zscale_contrast=.25),
                             MinMaxNormalizer(norm_min=0, norm_max=255.)])


def _check_catalog(plain, withm, img, header, x0=0, y0=0):
    from caesar_yolo_b200 import fits
    assert len(plain) == len(withm)
    for a, b in zip(plain, withm):
        assert {k: v for k, v in b.items() if k not in MKEYS} == a
        assert set(MKEYS) <= set(b)
    boxes = [(d['x1'], d['y1'], d['x2'], d['y2']) for d in withm]
    P, S, M = ref_measure(img, boxes)
    got = {k: np.array([np.nan if d[k] is None else d[k] for d in withm], np.float64) for k in MKEYS}
    np.testing.assert_array_equal(got['npix'], M['npix'])
    for k in ('peak', 'peak_x', 'peak_y'):
        np.testing.assert_array_equal(got[k], M[k], err_msg=k)
    assert np.all(np.abs(got['sum'] - P['sum']) <= 1e-12 * S['sum'])
    _close_derived(got, M, _moment_scale(P))
    beam = fits.beam_area_pix(header)
    if beam is None:
        assert all(d['flux'] is None for d in withm)
    else:
        np.testing.assert_allclose(got['flux'], P['sum'] / beam, rtol=1e-12, atol=1e-12 * S['sum'].max() / beam)
    radec = fits.pixel_to_world(header, M['xc'] + x0, M['yc'] + y0)
    if radec is None:
        assert all(d['ra'] is None and d['dec'] is None for d in withm)
    else:
        np.testing.assert_allclose(got['ra'], radec[0], rtol=0, atol=1e-9, equal_nan=True)
        np.testing.assert_allclose(got['dec'], radec[1], rtol=0, atol=1e-9, equal_nan=True)


def test_run_parallel_end_to_end(cuda_dev, tmp_path):
    from caesar_yolo_b200 import weights as W
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    img = synth.make_mosaic(1024, 1536, seed=3, nan_border_frac=0.01)
    path = str(tmp_path / "m.fits")
    synth.write_fits(path, img, WCS_CARDS)
    w = W.make_random_weights('n', 5, seed=0, cls_bias=-12.0)
    model = YOLO(w)
    cats = []
    for measure in (False, True):
        out = tmp_path / ("out%d" % measure)
        out.mkdir()
        sf = SFinder(model, _config(path, str(out), True, preprocess_fcn=_pp(True), measure_sources=measure))
        assert sf.run_parallel() == 0
        cats.append(json.load(open(str(out / "catalog_m.json")))['sources'])
        reg = open(str(out / "ds9_m.reg")).read()
        if measure:
            assert reg == plain_reg
        plain_reg = reg
    assert len(cats[0]) >= 10, "no detections: the test would be vacuous"
    _check_catalog(cats[0], cats[1], img, WCS_CARDS)
    assert any(d['ra'] is not None for d in cats[1]) and any(d['flux'] is not None for d in cats[1])


@pytest.mark.parametrize("crop", [False, True])
def test_run_serial_end_to_end(cuda_dev, tmp_path, crop):
    import os
    from caesar_yolo_b200 import fits, weights as W
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    img = np.load(os.path.join(os.path.dirname(__file__), "golden", "galaxy0001.npy")).astype(np.float32)
    if img.ndim == 3:
        img = img[..., 0]
    path = str(tmp_path / "g.fits")
    # whole image: no WCS / beam cards (flux, ra, dec are null); crop: the cards, so that ra / dec must use the file
    # pixel of the centroid (catalog pixel + crop offset)
    header = WCS_CARDS if crop else {}
    synth.write_fits(path, img, header)
    w = W.make_random_weights('n', 5, seed=0, cls_bias=-16.0)
    model = YOLO(w)
    ny, nx = img.shape
    x0, y0, x1, y1 = (nx // 8, ny // 6, nx - nx // 10, ny - ny // 7) if crop else (0, 0, nx, ny)
    kw = dict(image_xmin=x0, image_xmax=x1, image_ymin=y0, image_ymax=y1) if crop else {}
    objs = []
    for measure in (False, True):
        out = tmp_path / ("out%d" % measure)
        out.mkdir()
        sf = SFinder(model, _config(path, str(out), False, preprocess_fcn=_pp(False), measure_sources=measure, **kw))
        assert sf.run() == 0
        objs.append(json.load(open(str(out / "out_g.json")))['objs'])
    assert len(objs[0]) > 0, "no detections: the test would be vacuous"
    _check_catalog(objs[0], objs[1], img[y0:y1, x0:x1], header, x0, y0)
    if crop:   # the offset moves the sky position by more than the tolerance
        xc = np.array([d['xc'] for d in objs[1] if d['xc'] is not None])
        assert xc.size and np.all(np.abs(fits.pixel_to_world(header, xc + x0, 0 * xc)[0] -
                                         fits.pixel_to_world(header, xc, 0 * xc)[0]) > 1e-6)
