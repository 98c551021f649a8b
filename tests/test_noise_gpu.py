"""Local background and noise on the GPU (cy_noise_init / cy_noise_pass / cy_noise_update, SFinder with measure_noise)
against a numpy fp64 restatement of the definition in include/caesar_b200.h.

nbkg and iters are exact.  bkg is compared relative to |c| + mean |v - c| of its last pass, rms through its square
relative to mean (v - c)^2 + (mean (v - c))^2: the scales at which a reordered fp64 sum can differ.  A clip decision could
flip on such a difference only for a pixel that lies on a clip bound, so the restatement asserts that no kept pixel lies
within 1e-9 relative of a bound of its pass (a pixel equal to the mean sits at the centre of the interval and is exempt,
which covers the constant frame, whose sums are exact)."""
import json
import math

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import catalog, ops, synth

pytestmark = pytest.mark.gpu

F = 16
KAPPA, MAXITERS = 3.0, 5


def ref_noise(img, boxes, frame=F, r0=0, r1=None):
    """numpy restatement.  img: 2-D float32 (decoded values); boxes [n, 4] = x1, y1, x2, y2 inclusive; frames clipped to
    rows [r0, r1).  Returns a dict of arrays: bkg, rms, nbkg, iters and the comparison scales bkg_scale, var_scale."""
    ny, nx = img.shape
    r1 = ny if r1 is None else r1
    n = len(boxes)
    R = dict(bkg=np.full(n, np.nan), rms=np.full(n, np.nan), nbkg=np.zeros(n, np.int64), iters=np.zeros(n, np.int64),
             bkg_scale=np.zeros(n), var_scale=np.zeros(n))
    for i, (x1, y1, x2, y2) in enumerate(np.asarray(boxes, np.float64)):
        bx0, bx1, by0, by1 = math.ceil(x1), math.floor(x2), math.ceil(y1), math.floor(y2)
        if not (bx0 <= bx1 and by0 <= by1):
            continue
        gx0, gx1 = max(bx0 - frame, 0), min(bx1 + frame, nx - 1)
        gy0, gy1 = max(by0 - frame, r0), min(by1 + frame, r1 - 1)
        if gx0 > gx1 or gy0 > gy1:
            continue
        sub = img[gy0:gy1 + 1, gx0:gx1 + 1].astype(np.float64)
        with np.errstate(invalid='ignore'):
            keep = np.isfinite(sub) & (sub != 0)
        hy0, hy1, hx0, hx1 = max(by0, gy0), min(by1, gy1), max(bx0, gx0), min(bx1, gx1)
        if hy0 <= hy1 and hx0 <= hx1:
            keep[hy0 - gy0:hy1 - gy0 + 1, hx0 - gx0:hx1 - gx0 + 1] = False
        v = sub[keep]
        lo, hi, c, nprev = -np.inf, np.inf, 0.0, -1
        for k in range(MAXITERS + 1):
            kept = v[(v >= lo) & (v <= hi)]
            m = kept.size
            R['iters'][i] = k
            if m == 0:
                break
            d = kept - c
            s1, s2 = d.sum(), (d * d).sum()
            m1 = s1 / m
            mu = c + m1
            sd = math.sqrt(max(s2 / m - m1 * m1, 0.0))
            R['nbkg'][i], R['bkg'][i], R['rms'][i] = m, mu, sd
            R['bkg_scale'][i] = abs(c) + np.abs(d).sum() / m
            R['var_scale'][i] = s2 / m + m1 * m1
            if (k >= 1 and m == nprev) or k == MAXITERS:
                break
            for b in (mu - KAPPA * sd, mu + KAPPA * sd):
                near = (np.abs(kept - b) <= 1e-9 * (abs(mu) + KAPPA * sd)) & (kept != mu)
                assert not near.any(), ("fixture pixel on a clip bound", i, k)
            lo, hi, c, nprev = max(lo, mu - KAPPA * sd), min(hi, mu + KAPPA * sd), mu, m
    return R


def _src(boxes):
    s = np.zeros(len(boxes), dtype=ops.SRC_DTYPE)
    b = np.asarray(boxes, np.float32)
    s['x1'], s['y1'], s['x2'], s['y2'] = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    return s


def _gpu_noise(words, big_endian, ncols, boxes, ranges, dev, frame=F):
    """Every range is one rank with its own buffer (starting at its first row), state and unit plan; the partials of
    each pass are concatenated in range order, like the all-gather, and every rank folds them.  Asserts that the ranks
    agree on the active count and end with the same state.  -> (NOISE_DTYPE array, passes)."""
    src_dev = ops.to_device_bytes(_src(boxes), dev)
    n, world = len(boxes), len(ranges)
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ranks = []
    for r0, r1 in ranges:
        state = torch.empty((n * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
        off = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        units = ops.noise_init(src_dev, n, ncols, r0, r1, frame, state, off)
        ranks.append((full[r0:max(r1, r0 + 1)], r0, r1, state, off, units))
    active, passes = n, 0
    while active:
        parts = [ops.noise_pass(buf, ncols, big_endian, r0, ncols, src_dev, n, r0, r1, frame, off, units, state,
                                torch.empty((n * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev))
                 for buf, r0, r1, state, off, units in ranks]
        allp = torch.cat(parts)
        acts = {ops.noise_update(allp, world, n, r[3]) for r in ranks}
        assert len(acts) == 1
        active = acts.pop()
        passes += 1
        assert passes <= ops.NOISE_MAX_PASSES
    states = [r[3].cpu().numpy().view(ops.NOISE_DTYPE) for r in ranks]
    for s in states[1:]:
        assert s.tobytes() == states[0].tobytes()
    return states[0], passes


def _check(got, R):
    np.testing.assert_array_equal(got['nbkg'], R['nbkg'])
    np.testing.assert_array_equal(got['iters'], R['iters'])
    assert np.all(got['done'] == 1)
    ok = R['nbkg'] > 0
    np.testing.assert_array_equal(np.isnan(got['bkg']), ~ok)
    np.testing.assert_array_equal(np.isnan(got['rms']), ~ok)
    assert np.all(np.abs(got['bkg'][ok] - R['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
    assert np.all(np.abs(got['rms'][ok] ** 2 - R['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])


# ---------------------------------------------------------------------------------------------- fixtures

NY, NX = 2300, 2200
CONST_BOX = (320, 1520, 380, 1580)          # frame = 0.37 everywhere
SPECIAL_BOX = (1000, 1800, 1040, 1830)      # NaN, +-inf and 0 in its frame
NEIGHBOUR_BOX = (1500, 500, 1540, 540)      # a bright source 6 px right of the box, inside the frame
TAIL = (1800, 2000, 1200, 1500)             # rows, columns of a heavy-tailed (Student t, 1.5 dof) region


def _noise_mosaic(seed):
    img = synth.make_mosaic(NY, NX, seed=seed, nan_border_frac=0.0)   # edge frames hold pixels to clip
    rng = np.random.default_rng(seed + 100)
    img[2100:2200, 100:300] = np.nan                                    # all-NaN frames (and boxes) in here
    img[1504:1597, 304:397] = 0.37
    img[1520:1581, 320:381] = rng.standard_normal((61, 61)).astype(np.float32) * 1e-3 + 0.5   # the box itself
    img[1790, 1000:1010] = np.nan
    img[1795, 990:995] = np.inf
    img[1800:1805, 1045] = -np.inf
    img[1832:1840, 1020:1030] = 0.0
    yy, xx = np.mgrid[490:550, 1540:1560]
    img[490:550, 1540:1560] += (0.05 * np.exp(-0.5 * ((xx - 1548.3) ** 2 + (yy - 521.7) ** 2) / 2.0 ** 2)
                                ).astype(np.float32)
    y0, y1, x0, x1 = TAIL
    img[y0:y1, x0:x1] = (rng.standard_t(1.5, (y1 - y0, x1 - x0)) * 1e-3 + 2e-3).astype(np.float32)
    return img


def _noise_boxes(seed):
    nx, ny = NX, NY
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(-20, nx + 20, 300), rng.uniform(-20, ny + 20, 300)
    w, h = np.exp(rng.uniform(0, np.log(80), 300)), np.exp(rng.uniform(0, np.log(80), 300))
    b = np.floor(np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1))
    tail = [(x, y, x + 12, y + 10) for y in range(1830, 1960, 40) for x in range(1240, 1460, 50)]
    special = [
        (-15, -10, 30, 40), (nx - 5, -3, nx + 4, 12), (-4, ny - 6, 10, ny + 2), (nx - 20, ny - 8, nx + 30, ny + 5),
        (5, 800, 40, 830), (nx - 30, 900, nx - 8, 930), (700, 3, 740, 20), (800, ny - 12, 840, ny - 4),  # edges
        (nx + 3, 100, nx + 10, 120),                                    # box outside, frame inside the image
        (0, 0, nx - 1, ny - 1), (-5, -5, nx + 5, ny + 5),               # whole image: empty frame
        (5000, 10, 5010, 20), (50, 60, 40, 70),                         # far outside / empty box: empty frame
        CONST_BOX, SPECIAL_BOX, NEIGHBOUR_BOX,
        (80, 120, 2180, 2250),                                          # hull > 2000 x 2000
    ]
    return np.concatenate([b, np.asarray(tail + special, np.float64)])


def _special(boxes, box):
    return int(np.nonzero((boxes == np.asarray(box, np.float64)).all(1))[0][0])


@pytest.mark.parametrize("big_endian", [True, False])
def test_parity_with_numpy(cuda_dev, big_endian):
    img = _noise_mosaic(5)
    boxes = _noise_boxes(6)
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    got, passes = _gpu_noise(words, big_endian, NX, boxes, [(0, NY)], cuda_dev)
    R = ref_noise(img, boxes)
    _check(got, R)
    assert passes == R['iters'].max() + 1
    # the cases do what they say
    assert np.all(got['nbkg'][[_special(boxes, b) for b in ((0, 0, NX - 1, NY - 1), (-5, -5, NX + 5, NY + 5),
                                                            (5000, 10, 5010, 20), (50, 60, 40, 70))]] == 0)
    assert got['nbkg'][_special(boxes, (NX + 3, 100, NX + 10, 120))] > 0
    k = _special(boxes, CONST_BOX)
    assert got['rms'][k] == 0.0 and got['bkg'][k] == np.float64(np.float32(0.37)) and got['iters'][k] == 1
    k = _special(boxes, SPECIAL_BOX)
    x1, y1, x2, y2 = SPECIAL_BOX
    ring = img[y1 - F:y2 + F + 1, x1 - F:x2 + F + 1].astype(np.float64).copy()
    ring[F:-F, F:-F] = np.nan
    assert 0 < got['nbkg'][k] < np.sum(np.isfinite(ring) & (ring != 0)) + 1 and np.isfinite(got['bkg'][k])
    k = _special(boxes, NEIGHBOUR_BOX)
    assert got['iters'][k] >= 2 and abs(got['bkg'][k]) < 5e-5 and got['rms'][k] < 2e-4   # the neighbour is clipped
    assert np.any(got['iters'] == MAXITERS), "no source reaches the iteration cap: the case would be vacuous"
    assert got['nbkg'][_special(boxes, (80, 120, 2180, 2250))] > 50_000


def test_row_split_invariance(cuda_dev):
    img = _noise_mosaic(7)
    boxes = _noise_boxes(8)
    words = img.astype('>f4').view(np.int32)
    one, _ = _gpu_noise(words, True, NX, boxes, [(0, NY)], cuda_dev)
    R = ref_noise(img, boxes)
    _check(one, R)
    # NEIGHBOUR_BOX: frame-only rows 484..499 and 541..556, box rows 500..540; an empty range; the hull's frame rows
    for cuts in ([490], [520], [490, 520, 550], [1000, 1000, 2299], [100, 110, 2240, 2260], list(range(97, NY, 97))):
        edges = [0] + cuts + [NY]
        got, _ = _gpu_noise(words, True, NX, boxes, list(zip(edges[:-1], edges[1:])), cuda_dev)
        np.testing.assert_array_equal(got['nbkg'], one['nbkg'])
        np.testing.assert_array_equal(got['iters'], one['iters'])
        ok = one['nbkg'] > 0
        assert np.all(np.abs(got['bkg'][ok] - one['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
        assert np.all(np.abs(got['rms'][ok] ** 2 - one['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])
    # a run that measures only some rows clips the frames to them
    got, _ = _gpu_noise(words, True, NX, boxes, [(300, 1700)], cuda_dev)
    _check(got, ref_noise(img, boxes, r0=300, r1=1700))


def _measure(img_words, big_endian, ncols, boxes, rows, dev):
    src_dev = ops.to_device_bytes(_src(boxes), dev)
    full = torch.from_numpy(np.ascontiguousarray(img_words)).to(dev)
    part = ops.measure_sources(full, ncols, big_endian, 0, ncols, src_dev, len(boxes), rows[0], rows[1])
    return ops.measure_combine(part, 1, src_dev, len(boxes), ncols).cpu().numpy().view(ops.MEAS_DTYPE)


def test_physics_pedestal_and_noise(cuda_dev):
    """Gaussian noise sigma0 on a pedestal b0 with injected elliptical Gaussians: the frame statistics recover b0 and
    sigma0, and flux_bkgsub recovers the injected flux density where the raw flux is off by npix * b0 / A."""
    ny, nx = 700, 1000
    sigma0, b0, beam = 1e-3, 1e-2, 25.0
    rng = np.random.default_rng(11)
    img = b0 + sigma0 * rng.standard_normal((ny, nx))
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float64)
    cases = []   # x0, y0, amplitude, sigma_major, sigma_minor, theta (deg)
    for j, (x0, y0) in enumerate([(x, y) for y in (150.4, 350.7, 550.2) for x in (150.3, 400.6, 650.1, 850.8)]):
        cases.append((x0, y0, sigma0 * (30 + 40 * j), 2.0 + (j % 3), 1.5 + 0.3 * (j % 4), 25.0 * j))
    boxes = []
    for x0, y0, A, sa, sb, th in cases:
        t = math.radians(th)
        u = math.cos(t) * (xx - x0) + math.sin(t) * (yy - y0)
        v = -math.sin(t) * (xx - x0) + math.cos(t) * (yy - y0)
        img += A * np.exp(-0.5 * ((u / sa) ** 2 + (v / sb) ** 2))
        r = 6 * sa
        boxes.append((math.floor(x0 - r), math.floor(y0 - r), math.ceil(x0 + r), math.ceil(y0 + r)))
    img = img.astype(np.float32)
    words = img.view(np.int32)
    meas = _measure(words, False, nx, boxes, (0, ny), cuda_dev)
    noise, _ = _gpu_noise(words, False, nx, boxes, [(0, ny)], cuda_dev)
    _check(noise, ref_noise(img, boxes))
    d = catalog.measurement_dicts(meas, beam, None, noise)
    for m, z, dd, (x0, y0, A, sa, sb, th) in zip(meas, noise, d, cases):
        nb = int(z['nbkg'])
        assert abs(z['bkg'] - b0) <= 5 * sigma0 / math.sqrt(nb)
        # a Gaussian clipped at +-3 sigma converges to a std ~1.5 % below sigma0 (astropy applies no correction)
        assert abs(z['rms'] / sigma0 - 1) <= 5 / math.sqrt(2 * nb) + 0.02
        assert dd['snr'] == pytest.approx((m['peak'] - b0) / sigma0, rel=0.05)
        flux_true = 2 * math.pi * A * sa * sb / beam
        bias = int(m['npix']) * b0 / beam
        assert abs(dd['flux_bkgsub'] - flux_true) <= 5 * dd['flux_err']
        assert abs(dd['flux'] - flux_true) > 5 * dd['flux_err']                   # the bias this feature removes
        assert abs(dd['flux'] - flux_true - bias) <= 5 * dd['flux_err']


# ---------------------------------------------------------------------------------------------- end to end

WCS_CARDS = {"BMAJ": 0.0025, "BMIN": 0.002, "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN", "CRVAL1": 150.0,
             "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.0, "CDELT1": -0.0004, "CDELT2": 0.0004}


def _config(path, outdir, split, **kw):
    cfg = dict(img_size=640, preprocess_fcn=None, image_path=path, image_xmin=-1, image_xmax=-1, image_ymin=-1,
               image_ymax=-1, mpi=None, split_image_in_tiles=split, tile_xsize=512, tile_ysize=512, tile_xstep=1.0,
               tile_ystep=1.0, max_ntasks_per_worker=10000, devices=['cuda:0'], use_multi_gpu=False, iou_thr=0.5,
               merge_overlap_iou_thr_soft=0.3, merge_overlap_iou_thr_hard=0.8, score_thr=0.5, save_catalog=True,
               save_region=True, outdir=outdir)
    cfg.update(kw)
    return cfg


def _check_catalog(plain, noisy, img, header, r0, r1, frame):
    """plain: catalog of a measure_sources run; noisy: the same run with measure_noise."""
    from caesar_yolo_b200 import fits
    assert len(plain) == len(noisy) > 0
    for a, b in zip(plain, noisy):
        assert not set(catalog.NOISE_KEYS) & set(a)
        assert set(b) == set(a) | set(catalog.NOISE_KEYS)
        assert {k: b[k] for k in a} == a                       # the 13 measurement keys and the reference's keys
    boxes = [(d['x1'], d['y1'], d['x2'], d['y2']) for d in noisy]
    R = ref_noise(img, boxes, frame, r0, r1)
    got = np.zeros(len(noisy), dtype=ops.NOISE_DTYPE)
    for i, d in enumerate(noisy):
        got[i]['nbkg'] = d['nbkg']
        got[i]['bkg'] = np.nan if d['bkg'] is None else d['bkg']
        got[i]['rms'] = np.nan if d['rms'] is None else d['rms']
    got['iters'], got['done'] = R['iters'], 1    # iters is not written to the catalog
    _check(got, R)
    meas = np.zeros(len(noisy), dtype=ops.MEAS_DTYPE)
    for i, d in enumerate(noisy):
        meas[i]['npix'], meas[i]['sum'] = d['npix'], d['sum']
        meas[i]['peak'] = np.nan if d['peak'] is None else d['peak']
    want = [catalog.noise_keys(m, z, fits.beam_area_pix(header)) for m, z in zip(meas, got)]
    for d, w in zip(noisy, want):
        for k in ('snr', 'flux_bkgsub', 'flux_err'):
            assert (d[k] is None) == (w[k] is None), k
            if w[k] is not None:
                assert d[k] == pytest.approx(w[k], rel=1e-9, abs=1e-15), k
    assert any(d['snr'] is not None for d in noisy)


def test_run_parallel_end_to_end(cuda_dev, tmp_path):
    from caesar_yolo_b200 import weights as W
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    from caesar_yolo_b200.pipeline import measure_rows
    from caesar_yolo_b200.preprocessing import (BkgSubtractor, SigmaClipper, ChanResizer, ZScaleTransformer,
                                                Chan3Trasformer, MinMaxNormalizer, DataPreprocessor)
    pp = DataPreprocessor([BkgSubtractor(sigma=3), SigmaClipper(sigma_low=10, sigma_up=10), ChanResizer(nchans=3),
                           ZScaleTransformer(contrasts=[.25, .25, .25]),
                           Chan3Trasformer(sigma_clip_baseline=0, sigma_clip_low=10, sigma_clip_up=10,
                                           zscale_contrast=.25), MinMaxNormalizer(norm_min=0, norm_max=255.)])
    img = synth.make_mosaic(1024, 1536, seed=3, nan_border_frac=0.01)
    path = str(tmp_path / "m.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(W.make_random_weights('n', 5, seed=0, cls_bias=-12.0))
    cats, regs = [], []
    for noise in (False, True):
        out = tmp_path / ("out%d" % noise)
        out.mkdir()
        # measure_noise alone: it implies measure_sources
        kw = dict(measure_noise=True, noise_frame=12) if noise else dict(measure_sources=True)
        sf = SFinder(model, _config(path, str(out), True, preprocess_fcn=pp, **kw))
        assert sf.run_parallel() == 0
        cats.append(json.load(open(str(out / "catalog_m.json")))['sources'])
        regs.append(open(str(out / "ds9_m.reg")).read())
    assert regs[0] == regs[1]
    assert len(cats[0]) >= 10, "no detections: the test would be vacuous"
    tiles = sf.engine.tiles
    r0, r1 = measure_rows(tiles, 1)[0]
    _check_catalog(cats[0], cats[1], img, WCS_CARDS, r0, r1, 12)


def test_run_serial_crop_end_to_end(cuda_dev, tmp_path):
    import os
    from caesar_yolo_b200 import weights as W
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    from caesar_yolo_b200.preprocessing import ZScaleTransformer, MinMaxNormalizer, DataPreprocessor
    img = np.load(os.path.join(os.path.dirname(__file__), "golden", "galaxy0001.npy")).astype(np.float32)
    if img.ndim == 3:
        img = img[..., 0]
    path = str(tmp_path / "g.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(W.make_random_weights('n', 5, seed=0, cls_bias=-16.0))
    ny, nx = img.shape
    x0, y0, x1, y1 = nx // 8, ny // 6, nx - nx // 10, ny - ny // 7
    pp = DataPreprocessor([ZScaleTransformer(contrasts=[.25, .25, .25]), MinMaxNormalizer(norm_min=0, norm_max=255.)])
    objs = []
    for noise in (False, True):
        out = tmp_path / ("out%d" % noise)
        out.mkdir()
        kw = dict(measure_sources=True, measure_noise=noise)
        sf = SFinder(model, _config(path, str(out), False, preprocess_fcn=pp, image_xmin=x0, image_xmax=x1,
                                    image_ymin=y0, image_ymax=y1, **kw))
        assert sf.run() == 0
        objs.append(json.load(open(str(out / "out_g.json")))['objs'])
    # the frame is clipped to the crop: the restatement sees the cropped image only
    _check_catalog(objs[0], objs[1], img[y0:y1, x0:x1], WCS_CARDS, 0, y1 - y0, F)
