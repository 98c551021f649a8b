"""Source injection on the GPU (cy_inject_sources / cy_inject_restore / cy_bkg_grid_sample, SFinder with inject_sources)
against a numpy fp64 restatement of the definition in include/caesar_b200.h, and the properties the completeness
estimate rests on: the rows and records are restored bit for bit, a round's catalog is the catalog of a normal run on
the injected image, the injected S/N uses the rms map's bits, and no other output changes."""
import json
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import catalog, fits, inject, ops, synth
from caesar_yolo_b200.pipeline import Engine

pytestmark = pytest.mark.gpu

WCS = {"BMAJ": 0.0025, "BMIN": 0.002, "BPA": 30.0, "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN", "CRVAL1": 150.0,
       "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.0, "CDELT1": -0.0004, "CDELT2": 0.0004, "BUNIT": "JY/BEAM"}


def ref_inject(words, big_endian, row0, ncols, row_begin, row_end, inj, rx, ry, icov):
    """numpy fp64 restatement: words [rows, stride] uint32 (row 0 = image row row0) -> injected copy."""
    out = words.copy()
    ixx, ixy, iyy = icov
    dt = '>f4' if big_endian else '<f4'
    for q in inj:
        for y in range(q['cy'] - ry, q['cy'] + ry + 1):
            for x in range(q['cx'] - rx, q['cx'] + rx + 1):
                if x < 0 or x >= ncols or y < row_begin or y >= row_end:
                    continue
                v = words[y - row0, x:x + 1].view(dt)[0]
                if not np.isfinite(v) or v == 0:
                    continue
                dx, dy = float(x) - q['x'], float(y) - q['y']
                quad = (ixx * dx) * dx + ((2.0 * ixy) * dx) * dy + (iyy * dy) * dy
                o = np.float32(float(v) + q['peak'] * np.exp(-0.5 * quad))
                out[y - row0, x] = np.array([o], dt).view(np.uint32)[0]
    return out


@pytest.mark.parametrize("big_endian", [True, False])
def test_inject_kernel_and_restore(cuda_dev, big_endian):
    rng = np.random.default_rng(5)
    ny, stride, ncols, row0, rb, re = 120, 150, 140, 30, 38, 140
    img = rng.normal(1e-3, 2e-4, (ny, stride)).astype(np.float32)
    img[40:44, 60:70] = 0.0
    img[50, 60:66] = np.inf
    img[52, 61] = np.nan
    words = img.astype('>f4' if big_endian else '<f4').view(np.uint32)
    cov = fits.beam_cov_pix(WCS)
    rx, ry = inject.footprint_half(cov)
    icov = inject.inverse_cov(cov)
    # centres cut by column 0, column ncols (not the stride), row_begin, row_end, and one over the masked pixels
    cen = [(1.3, 60.2), (138.6, 80.7), (40.1, row0 + 9.4), (70.2, row0 + ny - 3.6), (63.4, 47.5), (100.0, 100.0)]
    inj = np.zeros(len(cen), ops.INJ_DTYPE)
    for k, (x, y) in enumerate(cen):
        inj[k] = (x, y, 5e-3 * (k + 1), int(np.floor(x + 0.5)), int(np.floor(y + 0.5)))
    dev = torch.from_numpy(words.view(np.int32).copy()).to(cuda_dev)
    eng = Engine.__new__(Engine)
    eng.device, eng._buf, eng.stage_events, eng.launches = cuda_dev, {}, None, 0
    h = eng.inject(dev, stride, big_endian, row0, ncols, rb, re, inj, rx, ry, icov)
    got = dev.cpu().numpy().view(np.uint32)
    want = ref_inject(words, big_endian, row0, ncols, rb, re, inj, rx, ry, icov)
    diff = got != want
    dt = '>f4' if big_endian else '<f4'
    ulps = np.abs(got.view(dt).astype(np.float32).view(np.int32).astype(np.int64)
                  - want.view(dt).astype(np.float32).view(np.int32).astype(np.int64))
    print("pixels off by one float32 ulp: %d of %d changed" % (int(diff.sum()), int((want != words).sum())))
    assert (ulps[diff] <= 1).all() and diff.sum() <= 8
    assert (want != words).sum() > 500
    masked = ~np.isfinite(img) | (img == 0)
    assert (got[masked] == words[masked]).all()
    assert (got[:, ncols:] == words[:, ncols:]).all() and (got[:rb - row0] == words[:rb - row0]).all()
    eng.restore(h)
    assert (dev.cpu().numpy().view(np.uint32) == words).all()


def test_bkg_grid_sample_is_the_map(cuda_dev):
    from test_bkgmap_gpu import NX, NY, _image
    img = _image(2)
    dev = torch.from_numpy(img.astype('>f4').view(np.int32)).to(cuda_dev)
    eng = Engine.__new__(Engine)
    eng.device, eng._buf, eng.stage_events, eng.launches = cuda_dev, {}, None, 0
    nodes, bkg, rms = eng.bkg_maps(dev, NX, True, 0, NX, 0, NY, 0, NY, box=31, grid=17)
    nodes2, b2, r2 = eng.bkg_maps(dev, NX, True, 0, NX, 0, NY, 0, NY, box=31, grid=17, maps=False)
    assert b2 is None and r2 is None and nodes.tobytes() == nodes2.tobytes()
    rng = np.random.default_rng(0)
    x, y = rng.integers(0, NX, 2000), rng.integers(0, NY, 2000)
    sb, sr = eng.sample_bkg_maps(nodes, NX, 0, NY, 31, 17, np.append(x, [-1, NX]), np.append(y, [0, 5]))
    mb = bkg.cpu().numpy().view('>f4').astype(np.float32)
    mr = rms.cpu().numpy().view('>f4').astype(np.float32)
    np.testing.assert_array_equal(sb[:-2].view(np.uint32), mb[y, x].view(np.uint32))
    np.testing.assert_array_equal(sr[:-2].view(np.uint32), mr[y, x].view(np.uint32))
    assert np.isnan(sb[-2:]).all() and np.isnan(sr[-2:]).all()


# ---------------------------------------------------------------------------------------------- end to end

def _config(path, outdir, split, **kw):
    cfg = dict(img_size=640, preprocess_fcn=None, image_path=path, image_xmin=-1, image_xmax=-1, image_ymin=-1,
               image_ymax=-1, mpi=None, split_image_in_tiles=split, tile_xsize=512, tile_ysize=512, tile_xstep=1.0,
               tile_ystep=1.0, max_ntasks_per_worker=10000, devices=['cuda:0'], use_multi_gpu=False, iou_thr=0.5,
               merge_overlap_iou_thr_soft=0.3, merge_overlap_iou_thr_hard=0.8, score_thr=0.5, save_catalog=True,
               save_region=True, outdir=outdir)
    cfg.update(kw)
    return cfg


def _pp():
    from caesar_yolo_b200.preprocessing import (BkgSubtractor, SigmaClipper, ChanResizer, ZScaleTransformer,
                                                Chan3Trasformer, MinMaxNormalizer, DataPreprocessor)
    return DataPreprocessor([BkgSubtractor(sigma=3), SigmaClipper(sigma_low=10, sigma_up=10), ChanResizer(nchans=3),
                             ZScaleTransformer(contrasts=[.25, .25, .25]),
                             Chan3Trasformer(sigma_clip_baseline=0, sigma_clip_low=10, sigma_clip_up=10,
                                             zscale_contrast=.25), MinMaxNormalizer(norm_min=0, norm_max=255.)])


@pytest.fixture(scope="module")
def model():
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.model import YOLO
    return YOLO(Wt.make_random_weights('n', 5, seed=0, cls_bias=-12.0))


@pytest.fixture(scope="module")
def mosaic(tmp_path_factory):
    img = synth.make_mosaic(1024, 1536, seed=3, nan_border_frac=0.01)
    img[600:606, 700:760] = 0.0
    path = str(tmp_path_factory.mktemp("inj") / "m.fits")
    synth.write_fits(path, img, WCS)
    return path, img


def _files(d):
    return {f: open(os.path.join(str(d), f), 'rb').read() for f in sorted(os.listdir(str(d)))}


class _Spy(object):
    """Records the rows each round injected into (a host copy taken right after cy_inject_sources) and the catalog of
    each round (the first argument of inject.match)."""

    def __init__(self, monkeypatch):
        self.rows, self.cats = [], []
        real_inject, real_match = Engine.inject, inject.match

        def spy_inject(eng, img, *a):
            h = real_inject(eng, img, *a)
            self.rows.append(img.cpu().numpy().copy())
            return h

        def spy_match(src, orig, cx, cy):
            self.cats.append(np.array(src, copy=True))
            return real_match(src, orig, cx, cy)
        monkeypatch.setattr(Engine, 'inject', spy_inject)
        monkeypatch.setattr(inject, 'match', spy_match)


def _injected_file(path, img, rows, r0, c0, out):
    """The FITS file of the original image with rows[r0:, c0:] written over it (big-endian words)."""
    words = img.astype('>f4').view(np.uint32).copy()
    words[r0:r0 + rows.shape[0], c0:c0 + rows.shape[1]] = rows.view(np.uint32)
    synth.write_fits_raw_be(out, words)
    return out


@pytest.mark.parametrize("step", [1.0, 0.5])
def test_round_catalog_is_a_run_on_the_injected_image(cuda_dev, tmp_path, monkeypatch, model, mosaic, step):
    """Key property: a round's catalog is byte for byte the catalog of a normal run_parallel on the injected image.
    Also: after the rounds the band holds the file's rows and a final exchange gives the original catalog."""
    from caesar_yolo_b200.inference import SFinder
    path, img = mosaic
    spy = _Spy(monkeypatch)
    out = tmp_path / "inj"
    out.mkdir()
    sf = SFinder(model, _config(path, str(out), True, preprocess_fcn=_pp(), tile_xstep=step, tile_ystep=step,
                                inject_sources=60, inject_rounds=2, inject_seed=11))
    assert sf.run_parallel() == 0
    doc = json.load(open(str(out / "inject_m.json")))
    assert [r['placed'] for r in doc['rounds']] == [60, 60] and len(spy.rows) == 2 and len(spy.cats) == 2
    orig = json.load(open(str(out / "catalog_m.json")))['sources']
    assert len(orig) >= 10, "no detections: the test would be vacuous"
    eng = sf.engine
    band, Y0, Y1, nx, _ = eng.band
    assert (band.cpu().numpy().view(np.uint32) == img[Y0:Y1].astype('>f4').view(np.uint32)).all()
    src, _ = eng.exchange_and_merge(1)
    assert catalog.sources_to_dicts(src, model.names) == orig
    for r in range(2):
        p = _injected_file(path, img, spy.rows[r], Y0, 0, str(tmp_path / ("r%d.fits" % r)))
        o2 = tmp_path / ("run%d" % r)
        o2.mkdir()
        sf2 = SFinder(model, _config(p, str(o2), True, preprocess_fcn=_pp(), tile_xstep=step, tile_ystep=step))
        assert sf2.run_parallel() == 0
        assert sf2.sources['sources'] == catalog.sources_to_dicts(spy.cats[r], model.names)
        changed = spy.rows[r].view(np.uint32) != img[Y0:Y1].astype('>f4').view(np.uint32)
        assert changed.sum() > 60 * 100
    print("rounds:", doc['rounds'], "recovered:", sum(d['recovered'] for d in doc['injections']))


def test_round_catalog_serial_crop(cuda_dev, tmp_path, monkeypatch, model, mosaic):
    from caesar_yolo_b200.inference import SFinder
    path, img = mosaic
    spy = _Spy(monkeypatch)
    x0, y0, x1, y1 = 113, 87, 811, 640
    out = tmp_path / "inj"
    out.mkdir()
    crop = dict(image_xmin=x0, image_xmax=x1, image_ymin=y0, image_ymax=y1, preprocess_fcn=_pp())
    sf = SFinder(model, _config(path, str(out), False, inject_sources=25, inject_rounds=2, **crop))
    assert sf.run() == 0
    doc = json.load(open(str(out / "inject_m.json")))
    assert [r['placed'] for r in doc['rounds']] == [25, 25]
    assert all(0 <= d['x'] < x1 - x0 and 0 <= d['y'] < y1 - y0 for d in doc['injections'])   # crop frame
    for r in range(2):
        p = _injected_file(path, img, spy.rows[r], y0, x0, str(tmp_path / ("r%d.fits" % r)))
        o2 = tmp_path / ("run%d" % r)
        o2.mkdir()
        sf2 = SFinder(model, _config(p, str(o2), False, **crop))
        assert sf2.run() == 0
        objs = json.load(open(str(o2 / ("out_r%d.json" % r))))['objs']
        want = [(o['x1'], o['y1'], o['x2'], o['y2'], o['score']) for o in objs]
        got = [tuple(float(s[k]) for k in ('x1', 'y1', 'x2', 'y2', 'score')) for s in spy.cats[r]]
        assert got == want


@pytest.mark.parametrize("est,mask", [('mean', False), ('mean', True), ('median', False), ('median', True)])
def test_rms_is_the_map_and_nothing_else_changes(cuda_dev, tmp_path, model, mosaic, est, mask):
    """rms in the JSON is the bits of rmsmap_<id>.fits at (c_x, c_y); the node states without the maps give the same
    JSON; with injection on every other file is byte for byte that of a run without it."""
    from caesar_yolo_b200.inference import SFinder
    path, img = mosaic
    opts = dict(preprocess_fcn=_pp(), bkg_estimator=est, bkg_mask_sources=mask, measure_noise=True,
                tile_xstep=0.5, tile_ystep=0.5)
    runs = {}
    for name, kw in (('maps', dict(save_bkg_maps=True, inject_sources=40)), ('plain', dict(save_bkg_maps=True)),
                     ('nomaps', dict(inject_sources=40))):
        out = tmp_path / name
        out.mkdir()
        assert SFinder(model, _config(path, str(out), True, **dict(opts, **kw))).run_parallel() == 0
        runs[name] = _files(out)
    inj = runs['maps'].pop('inject_m.json')
    assert runs['maps'] == runs['plain']
    assert runs['nomaps']['inject_m.json'] == inj
    doc = json.loads(inj)
    assert doc['params']['bkg_estimator'] == est and doc['params']['bkg_mask_sources'] is mask
    raw = runs['plain']['rmsmap_m.fits']
    H, W = img.shape
    n = len(fits.map_header(WCS, W, H, 0, 0, bkgmask=mask, bkgest=est))
    rms = np.frombuffer(raw[n:n + W * H * 4], '>u4').astype(np.uint32).reshape(H, W)
    assert len(doc['injections']) == 40
    for d in doc['injections']:
        cx, cy = int(np.floor(d['x'] + 0.5)), int(np.floor(d['y'] + 0.5))
        assert np.float32(d['rms']).view(np.uint32) == rms[cy, cx]
        assert d['peak'] == d['snr'] * d['rms']
