"""Reliability from the inverted image on the GPU (cy_negate_rows, cy_source_peak_snr, SFinder with reliability)
against numpy restatements of the definitions in include/caesar_b200.h, and the properties the estimate rests on: the
negation is exact and its own inverse, the bkg / rms / S/N maps are odd under it, the peak S/N is the maximum of the
S/N map's bytes over each box, the negative catalog is the catalog of a normal run on the inverted image, and no other
output changes."""
import json
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, ops, reliability, synth
from caesar_yolo_b200.pipeline import Engine
from test_bkgmap_gpu import NX, NY, _image
from test_inject_gpu import WCS, _config, _files, _pp, model, mosaic   # noqa: F401 (fixtures)
from test_snrmap_gpu import _gpu_snr

pytestmark = pytest.mark.gpu


def _bare_engine(dev):
    eng = Engine.__new__(Engine)
    eng.device, eng._buf, eng.stage_events, eng.launches = dev, {}, None, 0
    return eng


def ref_negate(words, big_endian, row0, ncols, row_begin, row_end):
    """numpy restatement: words [rows, stride] uint32 (row 0 = image row row0) -> negated copy."""
    out = words.copy()
    dec = words.byteswap() if big_endian else words
    mag = dec & np.uint32(0x7fffffff)
    flip = (mag != 0) & (mag < np.uint32(0x7f800000))
    rows = slice(row_begin - row0, row_end - row0)
    sign = np.uint32(0x80) if big_endian else np.uint32(0x80000000)
    blk = out[rows, :ncols]
    blk[flip[rows, :ncols]] ^= sign
    return out


# ---------------------------------------------------------------------------------------------- negation

@pytest.mark.parametrize("big_endian", [True, False])
def test_negate_rows_against_numpy(cuda_dev, big_endian):
    rng = np.random.default_rng(3)
    ny, stride = 70, 203
    img = rng.normal(0.0, 1.0, (ny, stride)).astype(np.float32)
    special = np.array([0.0, -0.0, np.nan, -np.nan, np.inf, -np.inf, 1e-45, -1e-45, 3.4e38, -3.4e38], np.float32)
    img[5:15, 20:30] = rng.choice(special, (10, 10))
    img[40, :] = -0.0
    words = img.astype('>f4' if big_endian else '<f4').view(np.uint32)
    words[7, 3] = np.uint32(0x7fc00123) if not big_endian else np.uint32(0x2301c07f)   # a NaN payload is kept
    eng = _bare_engine(cuda_dev)
    # crop column offsets of every alignment (the row starts are not 16-byte aligned), ncols < stride, rows inside
    for c0, ncols, row0, rb, re in ((0, 203, 0, 0, 70), (1, 150, 10, 12, 60), (2, 7, 3, 3, 40), (3, 1, 0, 30, 31),
                                    (5, 198, 20, 20, 20), (6, 3, 0, 0, 70)):
        dev = torch.from_numpy(words[row0:].view(np.int32).copy()).to(cuda_dev)
        eng.negate(dev[:, c0:], stride, big_endian, row0, ncols, rb, re)
        got = dev.cpu().numpy().view(np.uint32)
        want = words[row0:].copy()
        want[:, c0:] = ref_negate(np.ascontiguousarray(words[row0:, c0:]), big_endian, row0, ncols, rb, re)
        np.testing.assert_array_equal(got, want)
        eng.negate(dev[:, c0:], stride, big_endian, row0, ncols, rb, re)
        np.testing.assert_array_equal(dev.cpu().numpy().view(np.uint32), words[row0:])


def test_negate_refuses_bad_arguments(cuda_dev):
    dev = torch.zeros((4, 8), dtype=torch.int32, device=cuda_dev)
    for a in ((8, False, 0, 9, 0, 4), (8, False, 1, 8, 0, 4), (8, False, 0, 8, 3, 2), (8, False, 0, 0, 0, 4)):
        with pytest.raises(ops.CaesarB200Error):
            ops.negate_rows(dev, *a)
    ops.negate_rows(dev, 8, False, 0, 8, 2, 2)   # an empty row range is a no-op


# ---------------------------------------------------------------------------------------------- odd symmetry

@pytest.mark.parametrize("est", ['mean', 'median'])
@pytest.mark.parametrize("big_endian", [True, False])
def test_maps_are_odd_under_negation(cuda_dev, est, big_endian):
    """Without a mask, the maps of -I are -bkg and the same rms, and its S/N map is -snr, bit for bit (NaN borders
    and an all-masked block give NaN nodes)."""
    img = _image(11)
    words = img.astype('>f4' if big_endian else '<f4').view(np.uint32)
    eng = _bare_engine(cuda_dev)
    out = []
    for negate in (False, True):
        dev = torch.from_numpy(words.view(np.int32).copy()).to(cuda_dev)
        if negate:
            eng.negate(dev, NX, big_endian, 0, NX, 0, NY)
        nodes, bkg, rms = eng.bkg_maps(dev, NX, big_endian, 0, NX, 0, NY, 0, NY, box=51, grid=20, estimator=est)
        res, snr = eng.snr_maps(nodes, dev, NX, big_endian, 0, NX, 0, NY, 0, NY, box=51, grid=20)
        out.append((nodes.copy(), [t.cpu().numpy().view('>u4').astype(np.uint32) for t in (bkg, rms, res, snr)]))
    (n0, maps0), (n1, maps1) = out
    assert np.isnan(n0['bkg']).any() and np.isfinite(n0['bkg']).sum() > 100
    _odd(n0['bkg'], n1['bkg'])
    np.testing.assert_array_equal(n0['rms'].view(np.uint64), n1['rms'].view(np.uint64))
    b0, r0, s0, q0 = (m.view(np.float32) for m in maps0)
    b1, r1, s1, q1 = (m.view(np.float32) for m in maps1)
    np.testing.assert_array_equal(r1.view(np.uint32), r0.view(np.uint32))
    for a, b in ((b0, b1), (s0, s1), (q0, q1)):
        _odd(a, b)
    assert np.isfinite(q0).sum() > 0.5 * q0.size


def _odd(a, b):
    """b = -a: the same NaNs, and bit for bit elsewhere except that x - x is +0 in both images (a zero's sign)."""
    nan = np.isnan(a)
    np.testing.assert_array_equal(np.isnan(b), nan)
    np.testing.assert_array_equal(b[~nan], -a[~nan])
    nz = ~nan & (a != 0)
    np.testing.assert_array_equal(np.signbit(b[nz]), ~np.signbit(a[nz]))


# ---------------------------------------------------------------------------------------------- peak S/N

def ref_peak(snr, src, sign, X0, R0):
    """numpy restatement: snr float32 [H, W] (region columns from catalog column X0, rows from R0) -> (value, x, y)
    per source in catalog coordinates: the max of sign * snr over the integer box in the region, NaN skipped, -0 as +0,
    the first pixel in row-major order on ties."""
    H, W = snr.shape
    out_v, out_x, out_y = [], [], []
    for s in src:
        c = [float(s[k]) for k in ('x1', 'x2', 'y1', 'y2')]
        best = None
        if all(np.isfinite(c)):
            bx0, bx1 = max(int(np.ceil(c[0])), X0), min(int(np.floor(c[1])), X0 + W - 1)
            by0, by1 = max(int(np.ceil(c[2])), R0), min(int(np.floor(c[3])), R0 + H - 1)
            for y in range(by0, by1 + 1):
                for x in range(bx0, bx1 + 1):
                    v = snr[y - R0, x - X0]
                    if np.isnan(v):
                        continue
                    v = np.float32(-v) if sign < 0 else v
                    v = np.float32(0.0) if v == 0 else v
                    if best is None or v > best[0]:
                        best = (v, x, y)
        out_v.append(np.float32(np.nan) if best is None else best[0])
        out_x.append(-1 if best is None else best[1])
        out_y.append(-1 if best is None else best[2])
    return np.array(out_v, np.float32), np.array(out_x), np.array(out_y)


def _gpu_peak(words, big_endian, nodes, src, sign, box, grid, ranges, dev, X0=0, R0=0, W=None, H=None):
    """Peak S/N keys of one cy_source_peak_snr call per row range (each with its own buffer from its first row, as a
    rank's band), folded by their unsigned maximum and decoded."""
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ny_img, nx_img = words.shape
    W = nx_img - X0 if W is None else W
    H = ny_img - R0 if H is None else H
    st = ops.to_device_bytes(np.ascontiguousarray(nodes), dev)
    sd = ops.to_device_bytes(np.ascontiguousarray(src), dev)
    keys = np.zeros(len(src), np.uint64)
    for r0, r1 in ranges:
        out = torch.empty((len(src),), dtype=torch.int64, device=dev)
        ops.source_peak_snr(st, W, R0, R0 + H, box, grid, full[r0:max(r1, r0 + 1), X0:], nx_img, big_endian, r0, X0,
                            sd, len(src), sign, r0, r1, out)
        keys = np.maximum(keys, out.cpu().numpy().view(np.uint64))
    return ops.peak_snr_decode(keys, W, R0, X0)


def _sources(rng, n, X0, R0, W, H, extra=()):
    """Random integer-valued boxes around the region (some cut by its edges), plus `extra` (x1, y1, x2, y2)."""
    src = np.zeros(n + len(extra), ops.SRC_DTYPE)
    x = rng.integers(X0 - 20, X0 + W + 5, n)
    y = rng.integers(R0 - 20, R0 + H + 5, n)
    w, h = rng.integers(0, 40, n), rng.integers(0, 40, n)
    src['x1'][:n], src['y1'][:n], src['x2'][:n], src['y2'][:n] = x, y, x + w, y + h
    for k, b in enumerate(extra):
        src['x1'][n + k], src['y1'][n + k], src['x2'][n + k], src['y2'][n + k] = b
    src['score'] = 0.5
    return src


def _same_peaks(got, want):
    np.testing.assert_array_equal(got[0].view(np.uint32), want[0].view(np.uint32))
    np.testing.assert_array_equal(got[1], want[1])
    np.testing.assert_array_equal(got[2], want[2])


@pytest.mark.parametrize("est,mask", [('mean', False), ('mean', True), ('median', False), ('median', True)])
@pytest.mark.parametrize("sign", [1, -1])
def test_peak_snr_against_the_snr_map(cuda_dev, est, mask, sign):
    """Peak S/N of boxes in, across and outside a region with a column and row offset, against the max of the bytes of
    cy_bkg_grid_snr_maps over each box; invariant under splits of the rows into 1, 2 and 3 ranges."""
    big_endian = True
    img = _image(13)
    words = img.astype('>f4').view(np.int32)
    X0, R0, W, H = 23, 17, 560, 480
    rng = np.random.default_rng(4)
    extra = [(330, 230, 360, 260),                 # inside the NaN block: all masked
             (50.5, 60.5, 50.7, 80.0),             # empty integer box (ceil 51 > floor 50)
             (np.nan, 10, 20, 30),                 # NaN coordinates
             (X0 + W + 3, 100, X0 + W + 30, 140),  # right of the region
             (0, 0, X0 - 1, R0 - 1),               # left of and above the region
             (X0 + 100, R0 + 100, X0 + 100, R0 + 100)]   # one pixel
    src = _sources(rng, 300, X0, R0, W, H, extra)
    eng = _bare_engine(cuda_dev)
    full = torch.from_numpy(words.copy()).to(cuda_dev)
    region = full[:, X0:]
    m = None
    if mask:
        m = eng.source_mask(src, NX, R0, R0 + H)
    nodes = eng.bkg_maps(region[R0:], NX, big_endian, R0, W, R0, R0 + H, R0, R0 + H, box=51, grid=20, mask=m,
                         mask_col0=X0, estimator=est, maps=False)[0]
    _, snr = _gpu_snr(words, big_endian, nodes, 51, 20, [(R0, R0 + H)], cuda_dev, X0, R0, W, H)
    want = ref_peak(snr, src, sign, X0, R0)
    n_nan = int(np.isnan(want[0]).sum())
    assert 5 <= n_nan < len(src) // 2, n_nan
    got = eng.peak_snr(nodes, src, region[R0:], NX, big_endian, R0, W, R0, R0 + H, R0, R0 + H, 51, 20, col_off=X0,
                       sign=sign)
    _same_peaks(got, want)
    for cuts in ([R0 + 200], [R0 + 1, R0 + 333], [R0 + 100, R0 + 101]):
        edges = [R0] + cuts + [R0 + H]
        _same_peaks(_gpu_peak(words, big_endian, nodes, src, sign, 51, 20, list(zip(edges[:-1], edges[1:])),
                              cuda_dev, X0, R0, W, H), want)


@pytest.mark.parametrize("big_endian", [True, False])
def test_peak_snr_ties_and_node_rules(cuda_dev, big_endian):
    """Node states edited to bkg 1/4, rms 1 (snr = v - 1/4 exactly): ties of the largest value go to the first pixel in
    row-major order, -0 counts as +0; NaN, zero and negative rms nodes make the S/N NaN."""
    H, W = 120, 150
    rng = np.random.default_rng(9)
    img = rng.normal(0, 1, (H, W)).astype(np.float32)
    img[10:20, 10:20] = -1.0
    img[12, 15] = img[14, 11] = img[18, 19] = 7.0           # ties of the max (sign +1): (15, 12) wins
    img[30:40, 30:40] = 2.0
    img[33, 36] = img[31, 38] = -9.0                          # ties of the max of -snr: (38, 31) wins
    img[50:55, 50:55] = 1.0
    img[52, 53] = img[51, 54] = 0.25                          # snr +0; -snr -0, read as +0: (54, 51) wins
    img[50, 52] = 0.0                                         # masked
    nx_n, ny_n = len(ops.bkg_grid_nodes(W, 10)), len(ops.bkg_grid_nodes(H, 10))
    nodes = np.zeros((ny_n, nx_n), ops.NOISE_DTYPE)
    nodes['bkg'] = 0.25
    nodes['rms'] = 1.0
    nodes['rms'][8:10, 0:3] = np.nan
    nodes['rms'][10:12, 5:8] = 0.0
    nodes['rms'][0:2, 12:15] = -1.0
    words = img.astype('>f4' if big_endian else '<f4').view(np.int32)
    src = _sources(rng, 80, 0, 0, W, H, [(10, 10, 19, 19), (30, 30, 39, 39), (50, 50, 54, 54), (0, 80, 20, 90),
                                         (50, 100, 70, 110), (120, 0, 140, 10)])
    eng = _bare_engine(cuda_dev)
    dev = torch.from_numpy(words.copy()).to(cuda_dev)
    _, snr = _gpu_snr(words, big_endian, nodes, 11, 10, [(0, H)], cuda_dev)
    for sign in (1, -1):
        want = ref_peak(snr, src, sign, 0, 0)
        got = eng.peak_snr(nodes, src, dev, W, big_endian, 0, W, 0, H, 0, H, 11, 10, sign=sign)
        _same_peaks(got, want)
        _same_peaks(_gpu_peak(words, big_endian, nodes, src, sign, 11, 10, [(0, 13), (13, 31), (31, H)], cuda_dev),
                    want)
    p = eng.peak_snr(nodes, src, dev, W, big_endian, 0, W, 0, H, 0, H, 11, 10, sign=1)
    assert (p[0][-6], p[1][-6], p[2][-6]) == (6.75, 15, 12)
    assert (p[0][-4], p[1][-4], p[2][-4]) == (0.75, 50, 50)
    n = eng.peak_snr(nodes, src, dev, W, big_endian, 0, W, 0, H, 0, H, 11, 10, sign=-1)
    assert (n[0][-5], n[1][-5], n[2][-5]) == (9.25, 38, 31)
    assert (n[0][-4], n[1][-4], n[2][-4]) == (0.0, 54, 51) and not np.signbit(n[0][-4])
    # boxes whose pixels interpolate only NaN, zero or negative rms nodes
    assert np.isnan(p[0][-3:]).all() and np.isnan(n[0][-3:]).all() and (p[1][-3:] == -1).all()


def test_peak_snr_refuses_bad_arguments(cuda_dev):
    nodes = ops.to_device_bytes(np.zeros((2, 2), ops.NOISE_DTYPE), cuda_dev)
    img = torch.zeros((10, 10), dtype=torch.int32, device=cuda_dev)
    src = ops.to_device_bytes(np.zeros(1, ops.SRC_DTYPE), cuda_dev)
    out = torch.empty((1,), dtype=torch.int64, device=cuda_dev)
    for a in ((10, 0, 10, 3, 9, img, 10, False, 0, 0, src, 1, 0, 0, 10),      # sign 0
              (10, 0, 10, 3, 9, img, 10, False, 0, -1, src, 1, 1, 0, 10),     # negative column offset
              (10, 0, 10, 3, 9, img, 9, False, 0, 0, src, 1, 1, 0, 10),       # stride < ncols
              (10, 0, 10, 3, 9, img, 10, False, 0, 0, src, 1, 1, 0, 11),      # rows past the region
              (10, 0, 10, 4, 9, img, 10, False, 0, 0, src, 1, 1, 0, 10),      # even box
              (70000, 0, 70000, 3, 9, img, 70000, False, 0, 0, src, 1, 1, 0, 10)):   # 2^32 pixels or more
        with pytest.raises(ops.CaesarB200Error):
            ops.source_peak_snr(nodes, *a, out)


# ---------------------------------------------------------------------------------------------- end to end

def _negated_file(img, out):
    words = img.astype('>f4').view(np.uint32)
    synth.write_fits_raw_be(out, ref_negate(words, True, 0, words.shape[1], 0, words.shape[0]))
    return out


def _box_dicts(dicts):
    return [(d['x1'], d['y1'], d['x2'], d['y2'], d['class_name'], d['score']) for d in dicts]


def _check_tables(doc, cat_scores):
    lo, hi = doc['params']['snr_range']
    pos = np.array([np.nan if v is None else v for v in doc['catalog_snr_peak']], np.float64)
    neg = np.array([np.nan if d['snr_peak'] is None else d['snr_peak'] for d in doc['negative_detections']])
    edges = np.geomspace(lo, hi, 11)
    np.testing.assert_allclose(doc['params']['bin_edges'], edges, rtol=1e-15)
    for k, d in enumerate(doc['snr_cumulative']):
        assert d['n_pos'] == int((pos >= doc['params']['bin_edges'][k]).sum())
        assert d['n_neg'] == int((neg >= doc['params']['bin_edges'][k]).sum())
    assert sum(d['n_pos'] for d in doc['snr_bins']) == int(((pos >= lo) & (pos <= hi)).sum())
    assert sum(d['n_neg'] for d in doc['snr_bins']) == int(((neg >= lo) & (neg <= hi)).sum())
    assert doc['snr_outside']['nan'] == {'n_pos': int(np.isnan(pos).sum()), 'n_neg': int(np.isnan(neg).sum())}
    for d in doc['snr_bins'] + doc['snr_cumulative'] + doc['score_cumulative']:
        assert d['reliability'] == ((1 - d['n_neg'] / d['n_pos']) if d['n_pos'] else None)
    th = doc['params']['score_thresholds']
    sp, sn = np.array(cat_scores), np.array([d['score'] for d in doc['negative_detections']])
    assert [d['n_pos'] for d in doc['score_cumulative']] == [int((sp >= t).sum()) for t in th]
    assert [d['n_neg'] for d in doc['score_cumulative']] == [int((sn >= t).sum()) for t in th]
    t = reliability.tables(pos, neg, sp, sn, lo, hi, doc['params']['score_thr'])
    assert t['snr_bins'] == doc['snr_bins'] and t['snr_outside'] == doc['snr_outside']


def _peaks_against_map(doc, cat_dicts, snrmap_bytes, W, H, est, mask):
    n = len(fits.map_header(WCS, W, H, 0, 0, bkgmask=mask, bkgest=est, bunit=False))
    snr = np.frombuffer(snrmap_bytes[n:n + W * H * 4], '>u4').astype(np.uint32).view(np.float32).reshape(H, W)

    def src_of(dicts):
        s = np.zeros(len(dicts), ops.SRC_DTYPE)
        for k, d in enumerate(dicts):
            s[k]['x1'], s[k]['y1'], s[k]['x2'], s[k]['y2'] = d['x1'], d['y1'], d['x2'], d['y2']
        return s
    v, x, y = ref_peak(snr, src_of(cat_dicts), 1, 0, 0)
    assert [None if np.isnan(a) else float(a) for a in v] == doc['catalog_snr_peak']
    v, x, y = ref_peak(snr, src_of(doc['negative_detections']), -1, 0, 0)
    negs = doc['negative_detections']
    assert [None if np.isnan(a) else float(a) for a in v] == [d['snr_peak'] for d in negs]
    assert [None if a < 0 else int(a) for a in x] == [d['peak_x'] for d in negs]
    assert [None if a < 0 else int(a) for a in y] == [d['peak_y'] for d in negs]


@pytest.mark.parametrize("step,est,mask", [(1.0, 'mean', False), (0.5, 'median', True)])
def test_run_parallel_end_to_end(cuda_dev, tmp_path, model, mosaic, step, est, mask):
    from caesar_yolo_b200.inference import SFinder
    path, img = mosaic
    H, W = img.shape
    opts = dict(preprocess_fcn=_pp(), tile_xstep=step, tile_ystep=step, bkg_estimator=est, bkg_mask_sources=mask)
    runs = {}
    for name, kw in (('rel', dict(reliability=True, save_snr_maps=True)), ('plain', dict(save_snr_maps=True)),
                     ('relinj', dict(reliability=True, inject_sources=30)), ('inj', dict(inject_sources=30))):
        out = tmp_path / name
        out.mkdir()
        assert SFinder(model, _config(path, str(out), True, **dict(opts, **kw))).run_parallel() == 0
        runs[name] = _files(out)
    doc = json.loads(runs['rel'].pop('reliability_m.json'))
    reg = runs['rel'].pop('reliability_m.reg', None)
    assert runs['rel'] == runs['plain']
    assert json.loads(runs['relinj'].pop('reliability_m.json')) == doc      # node states without the maps
    runs['relinj'].pop('reliability_m.reg', None)
    assert runs['relinj'] == runs['inj']                                   # inject_m.json and the catalog unchanged
    # the negative catalog is the catalog of a normal run on the inverted image
    neg_path = _negated_file(img, str(tmp_path / "neg.fits"))
    out = tmp_path / "negrun"
    out.mkdir()
    sf = SFinder(model, _config(neg_path, str(out), True, preprocess_fcn=_pp(), tile_xstep=step, tile_ystep=step))
    assert sf.run_parallel() == 0
    negcat = json.load(open(str(out / "catalog_neg.json")))['sources']
    strip = [{k: v for k, v in d.items() if k not in ('snr_peak', 'peak_x', 'peak_y')}
             for d in doc['negative_detections']]
    assert strip == negcat
    assert len(negcat) >= 1, "no negative detections: the test would be vacuous"
    assert (reg is not None) == (len(negcat) > 0)
    cat = json.loads(runs['plain']['catalog_m.json'])['sources']
    assert doc['n_catalog'] == len(cat) and doc['n_negative'] == len(negcat)
    assert doc['params']['bkg_estimator'] == est and doc['params']['bkg_mask_sources'] is mask
    assert doc['n_tiles_rerun'] == len(ops.generate_tiles(0, W - 1, 0, H - 1, 512, 512, step, step))
    _peaks_against_map(doc, cat, runs['plain']['snrmap_m.fits'], W, H, est, mask)
    _check_tables(doc, [d['score'] for d in cat])
    print("catalog %d, negative %d, bins %s" % (len(cat), len(negcat), [d['n_pos'] for d in doc['snr_bins']]))


def test_run_serial_crop_end_to_end(cuda_dev, tmp_path, model, mosaic):
    from caesar_yolo_b200.inference import SFinder
    path, img = mosaic
    x0, y0, x1, y1 = 113, 87, 811, 640
    crop = dict(image_xmin=x0, image_xmax=x1, image_ymin=y0, image_ymax=y1, preprocess_fcn=_pp())
    runs = {}
    for name, kw in (('rel', dict(reliability=True)), ('plain', {})):
        out = tmp_path / name
        out.mkdir()
        assert SFinder(model, _config(path, str(out), False, **dict(crop, **kw))).run() == 0
        runs[name] = _files(out)
    doc = json.loads(runs['rel'].pop('reliability_m.json'))
    runs['rel'].pop('reliability_m.reg', None)
    assert runs['rel'] == runs['plain']
    neg_path = _negated_file(img, str(tmp_path / "neg.fits"))
    out = tmp_path / "negrun"
    out.mkdir()
    assert SFinder(model, _config(neg_path, str(out), False, **crop)).run() == 0
    objs = json.load(open(str(out / "out_neg.json")))['objs']
    assert _box_dicts(doc['negative_detections']) == _box_dicts(objs)
    cat = json.loads(runs['plain']['out_m.json'])['objs']
    assert doc['n_catalog'] == len(cat) and doc['n_tiles_rerun'] == 1
    assert all(d['peak_x'] is None or (0 <= d['peak_x'] < x1 - x0 and 0 <= d['peak_y'] < y1 - y0)
               for d in doc['negative_detections'])
    _check_tables(doc, [d['score'] for d in cat])
