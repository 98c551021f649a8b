"""Background-subtracted and S/N maps on the GPU (cy_bkg_grid_snr_maps, Engine.snr_maps, SFinder with save_snr_maps)
against a numpy fp64 restatement of the definition in include/caesar_b200.h, built from the node states and the bytes
of the bkg / rms maps: res = (float)(v - fb), snr = (float)((v - fb) / fr), with the NaN rules.  Every comparison is
exact to the float32 bit, NaN included."""
import json
import math
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, ops, synth
from test_bkgmap_gpu import _gpu_grid, _image, NY

pytestmark = pytest.mark.gpu

NAN32 = np.float32(np.nan)


def ref_res_snr(img, bkg, rms):
    """img: decoded float32 region; bkg, rms: the float32 values of the bkg / rms maps -> (res, snr) float32."""
    d = img.astype(np.float64) - bkg.astype(np.float64)
    fr = rms.astype(np.float64)
    with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
        res = d.astype(np.float32)
        snr = (d / np.where(fr > 0, fr, 1.0)).astype(np.float32)
        bad = ~np.isfinite(img) | (img == 0) | np.isnan(bkg)
        res[bad] = NAN32
        snr[bad | ~(fr > 0)] = NAN32
    return res, snr


def _bits(t):
    """Device rows of big-endian float32 words -> float32 array with the same bits (NaN payloads kept)."""
    return t.cpu().numpy().view('>u4').astype(np.uint32).view(np.float32)


def _same(got, want):
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


def _gpu_bkg(state, W, R0, R1, box, grid, dev):
    """bkg / rms maps of node states (numpy) over the whole region, as float32."""
    st = ops.to_device_bytes(np.ascontiguousarray(state), dev)
    b = torch.empty((R1 - R0, W), dtype=torch.int32, device=dev)
    r = torch.empty_like(b)
    ops.bkg_grid_maps(st, W, R0, R1, R0, R1, box, grid, b, r)
    return _bits(b), _bits(r)


def _gpu_snr(words, big_endian, nodes, box, grid, ranges, dev, X0=0, R0=0, W=None, H=None):
    """res / snr of the region (columns [X0, X0 + W), rows [R0, R0 + H) of the word array), one call per row range,
    each with its own buffer starting at its first row (as a rank's band) -> float32 [H, W] each."""
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ny_img, nx_img = words.shape
    W = nx_img - X0 if W is None else W
    H = ny_img - R0 if H is None else H
    st = ops.to_device_bytes(np.ascontiguousarray(nodes), dev)
    res, snr = [], []
    for r0, r1 in ranges:
        a = torch.empty((r1 - r0, W), dtype=torch.int32, device=dev)
        b = torch.empty_like(a)
        ops.bkg_grid_snr_maps(st, full[r0:max(r1, r0 + 1), X0:], nx_img, big_endian, r0, W, R0, R0 + H, r0, r1, box,
                              grid, a, b)
        res.append(_bits(a))
        snr.append(_bits(b))
    return np.concatenate(res), np.concatenate(snr)


def _check(img, words, big_endian, box, grid, dev, X0=0, R0=0, W=None, H=None, nodes=None):
    """Maps of the GPU nodes (or of `nodes`) against the restatement; returns (nodes, bkg, rms, res, snr)."""
    ny_img, nx_img = img.shape
    W = nx_img - X0 if W is None else W
    H = ny_img - R0 if H is None else H
    if nodes is None:
        nodes = _gpu_grid(words, big_endian, box, grid, [(R0, R0 + H)], dev, X0=X0, R0=R0, W=W, H=H)[0]
    bkg, rms = _gpu_bkg(nodes, W, R0, R0 + H, box, grid, dev)
    res, snr = _gpu_snr(words, big_endian, nodes, box, grid, [(R0, R0 + H)], dev, X0, R0, W, H)
    want = ref_res_snr(img[R0:R0 + H, X0:X0 + W], bkg, rms)
    _same(res, want[0])
    _same(snr, want[1])
    return nodes, bkg, rms, res, snr


@pytest.mark.parametrize("big_endian", [True, False])
def test_parity_with_numpy(cuda_dev, big_endian):
    """NaN borders, a NaN block (all-masked nodes), inf, -inf and 0 pixels, in both byte orders."""
    img = _image(5)
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    nodes, bkg, rms, res, snr = _check(img, words, big_endian, 51, 20, cuda_dev)
    bad = ~np.isfinite(img) | (img == 0)
    assert np.all(np.isnan(res[bad])) and np.all(np.isnan(snr[bad]))
    assert np.any(np.isnan(nodes['bkg'])) and np.isfinite(res).sum() > 0.5 * res.size


def test_nan_and_nonpositive_nodes(cuda_dev):
    """Node states edited so that every NaN rule is hit: NaN bkg (both maps NaN), NaN rms, rms 0 and rms < 0 (snr NaN,
    res finite)."""
    img = _image(8)
    words = img.astype('>f4').view(np.int32)
    nodes, _, _, _ = _gpu_grid(words, True, 51, 20, [(0, NY)], cuda_dev)
    nodes = nodes.copy()
    nodes['bkg'][3:6, 4:8] = np.nan           # a NaN bkg patch: the pixels between these nodes have no finite corner
    nodes['rms'][10:13, 10:14] = np.nan
    nodes['rms'][18:21, 2:6] = 0.0
    nodes['rms'][22:25, 20:24] = -1e-3
    _, bkg, rms, res, snr = _check(img, words, True, 51, 20, cuda_dev, nodes=nodes)
    fin = np.isfinite(img) & (img != 0)
    for cond in (np.isnan(bkg), np.isnan(rms), rms == 0, rms < 0):
        assert np.any(cond & fin), "a NaN rule is not exercised"
    assert np.all(np.isnan(res[np.isnan(bkg)]))
    assert np.all(np.isfinite(res[fin & ~np.isnan(bkg)]))
    assert np.all(np.isnan(snr[~(rms > 0)]))


def test_crop_offset(cuda_dev):
    img = _image(6)
    words = img.astype('>f4').view(np.int32)
    _check(img, words, True, 51, 20, cuda_dev, X0=37, R0=50, W=501, H=433)


def test_constant_image(cuda_dev):
    """rms = 0 everywhere: snr is NaN and res 0."""
    img = np.full((90, 130), 0.375, np.float32)
    _, bkg, rms, res, snr = _check(img, img.view(np.int32), False, 31, 10, cuda_dev)
    assert np.all(rms == 0) and np.all(res == 0) and not np.any(np.signbit(res)) and np.all(np.isnan(snr))


@pytest.mark.parametrize("H,W,box,grid", [
    (1, 200, 11, 7),       # one row: one node row
    (150, 1, 11, 7),       # one column
    (1, 1, 3, 1),          # one pixel: one node
    (60, 80, 21, 100),     # grid >= W and H: nodes on the corners only
    (40, 45, 301, 10),     # box larger than the image
    (77, 103, 3, 1),       # a node per pixel
])
def test_edge_lattices(cuda_dev, H, W, box, grid):
    rng = np.random.default_rng(H * 1000 + W)
    img = (rng.standard_normal((H, W)) * 1e-3 + 0.01).astype(np.float32)
    img[rng.random((H, W)) < 0.05] = np.nan
    _check(img, img.view(np.int32), False, box, grid, cuda_dev)


def test_row_split_invariance(cuda_dev):
    """Rows split over calls (each with its own buffer and row0) give the bytes of one call."""
    img = _image(7)
    words = img.astype('>f4').view(np.int32)
    nodes, _, _, res1, snr1 = _check(img, words, True, 101, 25, cuda_dev)
    for cuts in ([265], [100, 101], [0, 529], [13, 300, 301]):
        edges = [0] + cuts + [NY]
        res, snr = _gpu_snr(words, True, nodes, 101, 25, list(zip(edges[:-1], edges[1:])), cuda_dev)
        _same(res, res1)
        _same(snr, snr1)


def test_refuses_bad_arguments(cuda_dev):
    nodes = np.zeros((2, 2), dtype=ops.NOISE_DTYPE)
    st = ops.to_device_bytes(nodes, cuda_dev)
    img = torch.zeros((10, 10), dtype=torch.int32, device=cuda_dev)
    out = torch.empty((10, 10), dtype=torch.int32, device=cuda_dev)
    ok = dict(row_stride=10, row0=0, ncols=10, R0=0, R1=10, row_begin=0, row_end=10, box=11, grid=9)
    ops.bkg_grid_snr_maps(st, img, big_endian=False, res=out, snr=out.clone(), **ok)
    for bad in (dict(row_stride=9), dict(row0=1), dict(box=10), dict(box=1), dict(grid=0), dict(row_end=11),
                dict(row_begin=-1, row0=-1), dict(ncols=0)):
        with pytest.raises(ops.CaesarB200Error):
            ops.bkg_grid_snr_maps(st, img, big_endian=False, res=out, snr=out.clone(), **dict(ok, **bad))
    with pytest.raises(ops.CaesarB200Error):
        ops.bkg_grid_snr_maps(st, None, big_endian=False, res=out, snr=out.clone(), **ok)
    ops.bkg_grid_snr_maps(None, None, big_endian=False, res=None, snr=None, **dict(ok, row_end=0))   # no rows


def test_physics_pedestal_and_noise(cuda_dev):
    """Gaussian noise sigma0 on a pedestal b0 with one Gaussian source of peak A = 100 sigma0 on a pixel centre.  Away
    from the source, snr is standard normal: mean within 0.05 of 0 (the node bkg is off by ~sigma0 / 100) and std
    within 4 % of 1 (clipping at 3 sigma makes the node rms ~1.5 % low); the source's peak snr is A / sigma0 within 5 %
    (its own noise is sigma0, 1 %)."""
    H, W, s, A = 400, 450, 2.5, 100.0
    sigma0, b0 = 1e-3, 1e-2
    rng = np.random.default_rng(21)
    img = b0 + sigma0 * rng.standard_normal((H, W))
    yy, xx = np.mgrid[0:H, 0:W]
    r2 = (xx - 201.0) ** 2 + (yy - 187.0) ** 2
    img += A * sigma0 * np.exp(-0.5 * r2 / s ** 2)
    img = img.astype(np.float32)
    _, _, _, res, snr = _check(img, img.view(np.int32), False, 101, 25, cuda_dev)
    far = r2 > (8 * s) ** 2
    assert abs(float(snr[far].mean())) < 0.05
    assert abs(float(snr[far].std()) - 1.0) < 0.04
    assert abs(float(res[far].mean())) < 0.05 * sigma0
    assert abs(float(snr[187, 201]) / A - 1.0) < 0.05
    assert np.unravel_index(np.argmax(snr), snr.shape) == (187, 201)


# ---------------------------------------------------------------------------------------------- end to end

WCS_CARDS = {"BMAJ": 0.0025, "BMIN": 0.002, "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN", "CRVAL1": 150.0,
             "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.0, "CDELT1": -0.0004, "CDELT2": 0.0004,
             "BUNIT": "JY/BEAM"}
MAPS = ('bkgmap_', 'rmsmap_', 'resmap_', 'snrmap_')


def _config(path, outdir, split, **kw):
    cfg = dict(img_size=640, preprocess_fcn=None, image_path=path, image_xmin=-1, image_xmax=-1, image_ymin=-1,
               image_ymax=-1, mpi=None, split_image_in_tiles=split, tile_xsize=512, tile_ysize=512, tile_xstep=1.0,
               tile_ystep=1.0, max_ntasks_per_worker=10000, devices=['cuda:0'], use_multi_gpu=False, iou_thr=0.5,
               merge_overlap_iou_thr_soft=0.3, merge_overlap_iou_thr_hard=0.8, score_thr=0.5, save_catalog=True,
               save_region=True, outdir=outdir)
    cfg.update(kw)
    return cfg


def _files(d):
    return {f: open(os.path.join(str(d), f), 'rb').read() for f in sorted(os.listdir(str(d)))}


def _runs(tmp_path, run, make_sfinder, image_id, est, mask):
    """Runs: the bkg / rms maps alone; the S/N maps twice; none of the maps.  Checks the file sets and identities and
    returns (files of the S/N run, its SFinder)."""
    opts = dict(measure_sources=True, bkg_estimator=est, bkg_mask_sources=mask)
    kinds = [('bkg', dict(save_bkg_maps=True)), ('snr1', dict(save_snr_maps=True)), ('snr2', dict(save_snr_maps=True)),
             ('none', {})]
    files, sfs = {}, {}
    for name, kw in kinds:
        out = tmp_path / name
        out.mkdir()
        sf = make_sfinder(str(out), dict(opts, **kw))
        assert run(sf) == 0
        files[name], sfs[name] = _files(out), sf
    bkg_names, snr_names = ({p + image_id + '.fits' for p in ps} for ps in (MAPS[:2], MAPS[2:]))
    assert files['snr1'] == files['snr2']
    assert bkg_names <= set(files['bkg']) and not snr_names & set(files['bkg'])
    assert set(files['snr1']) == set(files['bkg']) | snr_names
    assert set(files['none']) == set(files['bkg']) - bkg_names
    for f in files['bkg']:   # the bkg / rms maps and the catalog are those of the run without the option
        assert files['bkg'][f] == files['snr1'][f], f
    return files['snr1'], sfs['snr1']


def _check_files(files, image_id, region_img, X0, R0, est, mask):
    """Headers of the four maps and res / snr against the restatement from the bkg / rms map bytes of the same run."""
    H, W = region_img.shape
    dec = {}
    for p in MAPS:
        raw = files[p + image_id + '.fits']
        hdr = fits.map_header(WCS_CARDS, W, H, X0, R0, bkgmask=mask, bkgest=est, bunit=p != 'snrmap_')
        assert raw[:len(hdr)] == hdr, p
        assert len(raw) % 2880 == 0 and raw[len(hdr) + W * H * 4:] == b'\0' * (len(raw) - len(hdr) - W * H * 4)
        dec[p] = np.frombuffer(raw[len(hdr):len(hdr) + W * H * 4], '>u4').astype(np.uint32).view(np.float32) \
            .reshape(H, W)
    res, snr = ref_res_snr(region_img, dec['bkgmap_'], dec['rmsmap_'])
    _same(dec['resmap_'], res)
    _same(dec['snrmap_'], snr)
    return dec


def _in_boxes(objs, dec, x_off=0, y_off=0):
    """The source mask is not applied to res / snr: the data pixels of the catalog boxes are finite there."""
    n = 0
    for d in objs:
        xa, xb = int(math.ceil(d['x1'])) - x_off, int(math.floor(d['x2'])) - x_off
        ya, yb = int(math.ceil(d['y1'])) - y_off, int(math.floor(d['y2'])) - y_off
        sub = dec['snrmap_'][max(ya, 0):yb + 1, max(xa, 0):xb + 1]
        n += int(np.isfinite(sub).sum())
    return n


CASES = [('mean', False), ('mean', True), ('median', False), ('median', True)]


@pytest.mark.parametrize("est,mask", CASES)
def test_run_parallel_end_to_end(cuda_dev, tmp_path, est, mask):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    from caesar_yolo_b200.preprocessing import (BkgSubtractor, SigmaClipper, ChanResizer, ZScaleTransformer,
                                                Chan3Trasformer, MinMaxNormalizer, DataPreprocessor)
    pp = DataPreprocessor([BkgSubtractor(sigma=3), SigmaClipper(sigma_low=10, sigma_up=10), ChanResizer(nchans=3),
                           ZScaleTransformer(contrasts=[.25, .25, .25]),
                           Chan3Trasformer(sigma_clip_baseline=0, sigma_clip_low=10, sigma_clip_up=10,
                                           zscale_contrast=.25), MinMaxNormalizer(norm_min=0, norm_max=255.)])
    img = synth.make_mosaic(1024, 1536, seed=3, nan_border_frac=0.01)
    path = str(tmp_path / "m.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(Wt.make_random_weights('n', 5, seed=0, cls_bias=-12.0))
    files, sf = _runs(tmp_path, lambda s: s.run_parallel(),
                      lambda out, kw: SFinder(model, _config(path, out, True, preprocess_fcn=pp, **kw)), 'm', est, mask)
    eng = sf.engine
    nodes, _, _, (X0, R0, W, H), rows = eng.bkg_maps_band(eng.tiles, estimator=est)
    assert (X0, R0, W, H) == (0, 0, 1536, 1024) and rows == (0, 1024)
    dec = _check_files(files, 'm', img, X0, R0, est, mask)
    objs = json.loads(files['catalog_m.json'])['sources']
    assert len(objs) >= 10, "no detections: the test would be vacuous"
    assert _in_boxes(objs, dec) > 0
    if not mask:   # Engine.snr_maps_band of the run's nodes gives the file bytes
        res, snr, region, rows2 = eng.snr_maps_band(nodes, eng.tiles)
        assert region == (X0, R0, W, H) and rows2 == rows
        n = len(fits.map_header(WCS_CARDS, W, H, X0, R0, bkgest=est, bunit=False))
        assert files['snrmap_m.fits'][n:n + W * H * 4] == snr.cpu().numpy().tobytes()
        n = len(fits.map_header(WCS_CARDS, W, H, X0, R0, bkgest=est))
        assert files['resmap_m.fits'][n:n + W * H * 4] == res.cpu().numpy().tobytes()
        with pytest.raises(ops.CaesarB200Error):   # node states of another lattice
            eng.snr_maps_band(nodes[:-1], eng.tiles)


@pytest.mark.parametrize("est,mask", CASES)
def test_run_serial_crop_end_to_end(cuda_dev, tmp_path, est, mask):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    img = synth.make_mosaic(700, 900, seed=4, nan_border_frac=0.02)
    img[300:305, 400:420] = 0.0
    img[310, 410:415] = np.inf
    path = str(tmp_path / "g.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(Wt.make_random_weights('n', 5, seed=0, cls_bias=-12.0))
    x0, y0, x1, y1 = 113, 87, 811, 640
    files, sf = _runs(tmp_path, lambda s: s.run(),
                      lambda out, kw: SFinder(model, _config(path, out, False, image_xmin=x0, image_xmax=x1,
                                                             image_ymin=y0, image_ymax=y1, bkg_box=51, bkg_grid=20,
                                                             **kw)), 'g', est, mask)
    dec = _check_files(files, 'g', img[y0:y1, x0:x1], x0, y0, est, mask)
    assert np.isnan(dec['snrmap_'][300 - y0, 400 - x0]) and np.isnan(dec['resmap_'][310 - y0, 410 - x0])
    objs = json.loads(files['out_g.json'])['objs']
    if objs:
        assert _in_boxes(objs, dec) > 0
