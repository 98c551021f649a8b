"""CPU tests of the host side of the source injection (inject_sources): the pixel covariance of the beam, the
placement rules, the affected tiles, the matching and the completeness bins, and the option surface (config, CLI,
SFinder checks, the PNG warning, no file with the option off)."""
import importlib.util
import json
import logging
import math
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, inject, ops, synth
from caesar_yolo_b200.config import CONFIG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 2.0 * math.sqrt(2.0 * math.log(2.0))


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_inject", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _Model:
    names = {0: 'a', 1: 'b'}


# ---------------------------------------------------------------------------------------------- beam covariance

@pytest.mark.parametrize("bpa,want", [
    (0.0, lambda sj, sn: [[sn, 0.0], [0.0, sj]]),            # major axis north = +y
    (90.0, lambda sj, sn: [[sj, 0.0], [0.0, sn]]),           # major axis east: along x, whatever the sign of CDELT1
    (30.0, lambda sj, sn: [[0.25 * sj + 0.75 * sn, -(sj - sn) * 0.5 * math.sqrt(3) / 2],
                           [-(sj - sn) * 0.5 * math.sqrt(3) / 2, 0.75 * sj + 0.25 * sn]]),
])
def test_cov_cdelt(bpa, want):
    """CDELT1 = -a, CDELT2 = a: C_pix = diag(-1/a, 1/a) C_sky diag(-1/a, 1/a); at BPA 30 the major axis (sin 30, cos 30)
    (east of north) points to -x, +y in pixels, so C_xy < 0."""
    a, bmaj, bmin = 4e-4, 2.5e-3, 2e-3
    c = fits.beam_cov_pix({"BMAJ": bmaj, "BMIN": bmin, "BPA": bpa, "CDELT1": -a, "CDELT2": a})
    sj, sn = (bmaj / K / a) ** 2, (bmin / K / a) ** 2
    np.testing.assert_allclose(c, want(sj, sn), rtol=1e-12, atol=1e-12 * sj)


def test_cov_bpa_default_is_zero():
    h = {"BMAJ": 2.5e-3, "BMIN": 2e-3, "CDELT1": -4e-4, "CDELT2": 4e-4}
    np.testing.assert_array_equal(fits.beam_cov_pix(h), fits.beam_cov_pix(dict(h, BPA=0.0)))


def test_cov_rotated_cd():
    """A rotated, sheared CD matrix: M C_pix M^T = C_sky, and the CROTA2 form of the same matrix gives the same C_pix.
    With CROTA2 = rho (M = a R(rho) diag(-1, 1), C&G eq. 189) the beam of position angle BPA lies on the pixel grid as
    that of BPA + rho on an unrotated grid."""
    bmaj, bmin, bpa = 3e-3, 1e-3, 40.0
    cd = np.array([[-3.9e-4, 0.7e-4], [0.5e-4, 4.1e-4]])
    h = {"BMAJ": bmaj, "BMIN": bmin, "BPA": bpa, "CD1_1": cd[0, 0], "CD1_2": cd[0, 1], "CD2_1": cd[1, 0],
         "CD2_2": cd[1, 1]}
    c = fits.beam_cov_pix(h)
    p = math.radians(bpa)
    u, v = np.array([math.sin(p), math.cos(p)]), np.array([math.cos(p), -math.sin(p)])
    c_sky = (bmaj / K) ** 2 * np.outer(u, u) + (bmin / K) ** 2 * np.outer(v, v)
    np.testing.assert_allclose(cd @ c @ cd.T, c_sky, rtol=1e-10, atol=1e-22)
    a, rho = 4e-4, 25.0
    rot = {"BMAJ": bmaj, "BMIN": bmin, "CDELT1": -a, "CDELT2": a, "CROTA2": rho}
    m = fits.pixel_scale_matrix(rot)
    h_cd = dict(rot, BPA=bpa, CD1_1=m[0, 0], CD1_2=m[0, 1], CD2_1=m[1, 0], CD2_2=m[1, 1])
    np.testing.assert_allclose(fits.beam_cov_pix(h_cd), fits.beam_cov_pix(dict(rot, BPA=bpa)), rtol=1e-12)
    np.testing.assert_allclose(fits.beam_cov_pix(dict(rot, BPA=bpa)),
                               fits.beam_cov_pix({"BMAJ": bmaj, "BMIN": bmin, "BPA": bpa + rho, "CDELT1": -a,
                                                  "CDELT2": a}), rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("h", [{}, {"BMAJ": 1e-3, "BMIN": 1e-3}, {"CDELT1": -1e-4, "CDELT2": 1e-4},
                               {"BMAJ": 1e-3, "CDELT1": -1e-4, "CDELT2": 1e-4},
                               {"BMAJ": 0.0, "BMIN": 1e-3, "CDELT1": -1e-4, "CDELT2": 1e-4},
                               {"BMAJ": 1e-3, "BMIN": 1e-3, "CDELT1": 0.0, "CDELT2": 1e-4}])
def test_cov_without_beam_or_scale(h):
    assert fits.beam_cov_pix(h) is None


def test_footprint_and_inverse():
    c = [[2.25, 0.5], [0.5, 4.0]]
    assert inject.footprint_half(c) == (6, 8)
    ixx, ixy, iyy = inject.inverse_cov(c)
    np.testing.assert_allclose(np.array([[ixx, ixy], [ixy, iyy]]) @ np.array(c), np.eye(2), atol=1e-15)


def _header_fits(path, beam=True):
    cards = {"CDELT1": -4e-4, "CDELT2": 4e-4}
    if beam:
        cards.update(BMAJ=2.5e-3, BMIN=2e-3)
    synth.write_fits(path, np.ones((64, 80), np.float32), cards)


@pytest.mark.parametrize("tiled", [False, True])
def test_no_beam_is_an_error_before_any_tile(tmp_path, caplog, tiled):
    from caesar_yolo_b200.inference import SFinder
    path = str(tmp_path / "n.fits")
    _header_fits(path, beam=False)
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(tmp_path), inject_sources=4, image_xmin=-1,
                                image_xmax=-1, image_ymin=-1, image_ymax=-1, tile_xsize=32, tile_ysize=32))
    sf._engine = None   # any engine use (a processed tile) would raise
    caplog.set_level(logging.ERROR)
    assert (sf.run_parallel() if tiled else sf.run()) == -1
    assert any('beam' in r.getMessage() for r in caplog.records)
    assert os.listdir(str(tmp_path)) == ['n.fits']


# ---------------------------------------------------------------------------------------------- placement

REGION = (10, 20, 300, 200)


def _place(seed=7, rnd=0, n=30, boxes=None, masked=None, rms=None, region=REGION, rx=3, ry=4, rng=(3.0, 100.0)):
    boxes = boxes if boxes is not None else tuple(np.zeros(0, np.int64) for _ in range(4))
    masked = masked or (lambda cx, cy: np.zeros(len(cx), bool))
    rms = rms or (lambda cx, cy: np.full(len(cx), 0.5, np.float32))
    return inject.place(seed, rnd, n, region, rx, ry, boxes, masked, rms, rng)


def test_placement_is_deterministic_and_seeded():
    a, b = _place(), _place()
    for k in ('x', 'y', 'cx', 'cy', 'snr', 'rms', 'peak'):
        np.testing.assert_array_equal(a[k], b[k])
    assert a['rejected'] == b['rejected'] and len(a['x']) == 30
    c, d = _place(seed=8), _place(rnd=1)
    assert not np.array_equal(a['x'], c['x']) and not np.array_equal(a['x'], d['x'])
    u = np.random.default_rng([7, 0]).random((600, 3))   # the first candidate, when it is accepted
    assert a['x'][0] == REGION[0] - 0.5 + u[0, 0] * REGION[2] or a['rejected']['outside'] > 0


def test_placement_rules():
    """Every rule rejects and no accepted injection breaks one."""
    rx, ry = 3, 4
    X0, R0, W, H = REGION
    bx = (np.array([100, 200]), np.array([140, 230]), np.array([50, 120]), np.array([90, 170]))

    def masked(cx, cy):
        return (cx % 7) == 0

    def rms(cx, cy):
        r = np.full(len(cx), 0.5, np.float32)
        r[(cy % 11) == 0] = np.nan
        r[(cy % 13) == 0] = 0.0
        r[(cy % 17) == 0] = -1.0
        return r
    p = _place(n=400, boxes=bx, masked=masked, rms=rms, rx=rx, ry=ry)
    assert all(p['rejected'][k] > 0 for k in inject.REJECT_RULES), p['rejected']
    cx, cy = p['cx'], p['cy']
    assert ((cx - rx >= X0) & (cx + rx <= X0 + W - 1) & (cy - ry >= R0) & (cy + ry <= R0 + H - 1)).all()
    assert not masked(cx, cy).any() and (rms(cx, cy) > 0).all()
    for b0, b1, c0, c1 in zip(*bx):
        assert not ((cx + rx >= b0) & (cx - rx <= b1) & (cy + ry >= c0) & (cy - ry <= c1)).any()
    d = (np.abs(cx[:, None] - cx[None, :]) <= 2 * rx) & (np.abs(cy[:, None] - cy[None, :]) <= 2 * ry)
    assert d.sum() == len(cx)   # disjoint footprints: only the diagonal
    assert np.array_equal(p['peak'], p['snr'] * p['rms'].astype(np.float64))
    assert ((p['snr'] >= 3.0) & (p['snr'] <= 100.0)).all()
    assert np.array_equal(np.floor(p['x'] + 0.5), cx) and np.array_equal(np.floor(p['y'] + 0.5), cy)


def test_placement_count_cap():
    """A region with room for few footprints: 20 N candidates are drawn, fewer than N placed."""
    p = _place(n=50, region=(0, 0, 30, 30), rx=4, ry=4)
    assert p['drawn'] == 20 * 50 and 0 < len(p['x']) < 50
    assert sum(p['rejected'].values()) == p['drawn'] - len(p['x'])
    q = _place(n=5, region=(0, 0, 5, 5), rx=4, ry=4)   # no footprint fits
    assert len(q['x']) == 0 and q['rejected']['outside'] == 100


def test_placement_log_uniform_snr():
    p = _place(n=2000, region=(0, 0, 4000, 4000), rx=1, ry=1, rng=(2.0, 200.0))
    frac = np.histogram(np.log10(p['snr']), bins=4, range=(math.log10(2), math.log10(200)))[0] / len(p['snr'])
    assert np.abs(frac - 0.25).max() < 0.05
    q = _place(n=10, rng=(5.0, 5.0))
    assert (q['snr'] == 5.0).all()


# ---------------------------------------------------------------------------------------------- affected tiles

@pytest.mark.parametrize("step", [1.0, 0.5])
def test_affected_tiles_brute_force(step):
    tiles = ops.generate_tiles(0, 999, 0, 799, 128, 96, step, step)
    rng = np.random.default_rng(3)
    cx, cy = rng.integers(-5, 1005, 60), rng.integers(-5, 805, 60)
    rx, ry = 5, 3
    want = []
    for t, tl in enumerate(tiles):
        px = np.zeros((800 + 20, 1000 + 20), bool)   # pixels of the tile, brute force
        px[tl['ymin'] + 10:tl['ymax'] + 10, tl['xmin'] + 10:tl['xmax'] + 10] = True
        if any(px[max(y - ry + 10, 0):y + ry + 11, max(x - rx + 10, 0):x + rx + 11].any() for x, y in zip(cx, cy)):
            want.append(t)
    got = inject.affected_tiles(tiles, cx, cy, rx, ry, chunk=7)
    assert got.tolist() == want and 0 < len(want) < len(tiles)
    assert len(inject.affected_tiles(tiles, [], [], rx, ry)) == 0


# ---------------------------------------------------------------------------------------------- matching, bins

def _src(rows):
    s = np.zeros(len(rows), ops.SRC_DTYPE)
    for i, (x1, y1, x2, y2, score, cls) in enumerate(rows):
        s[i] = (x1, y1, x2, y2, score, cls, 0, i)
    return s


def test_match_new_lost():
    orig = _src([(10, 10, 20, 20, .9, 0), (50, 50, 60, 60, .8, 1), (80, 80, 90, 90, .7, 0)])
    rnd = np.concatenate([orig[:1], orig[2:],   # source 1 is lost
                          _src([(99.5, 99.5, 110, 110, .75, 1),      # box [100, 110]: contains (100, 100)
                                (98, 98, 112, 112, .72, 0),          # also contains it, later in catalog order
                                (200, 200, 210, 210, .71, 0)])])     # new: matches nothing
    idx, new, lost = inject.match(rnd, orig, np.array([100, 99, 300]), np.array([100, 100, 300]))
    assert idx.tolist() == [2, 3, -1]   # (99, 100): outside [100, 110], inside [98, 112]
    assert new == 1 and lost == 1
    idx, new, lost = inject.match(orig, orig, np.array([15]), np.array([15]))
    assert idx.tolist() == [0] and new == 0 and lost == 0


def test_match_integer_box_edges():
    s = _src([(10.2, 10.0, 19.8, 20.0, .9, 0)])   # integer box [11, 19] x [10, 20]
    idx, _, _ = inject.match(s, s[:0], np.array([10, 11, 19, 20, 15, 15]), np.array([15, 15, 15, 15, 10, 21]))
    assert idx.tolist() == [-1, 0, 0, -1, 0, -1]


def test_completeness_bins():
    lo, hi = 3.0, 300.0
    snr = np.array([3.0, 3.5, 4.7, 30.0, 299.0, 300.0])
    rec = np.array([True, False, True, True, False, True])
    b = inject.completeness(snr, rec, lo, hi)
    assert len(b) == 10 and b[0]['snr_lo'] == pytest.approx(3.0) and b[-1]['snr_hi'] == pytest.approx(300.0)
    # edges 3 * 10^(k / 5): 3.0, 3.5 -> bin 0; 4.7 -> bin 0 (< 4.75); 30 -> bin 5; 299, 300 -> bin 9
    assert [d['n'] for d in b] == [3, 0, 0, 0, 0, 1, 0, 0, 0, 2]
    assert [d['recovered'] for d in b] == [2, 0, 0, 0, 0, 1, 0, 0, 0, 1]
    assert b[0]['fraction'] == pytest.approx(2 / 3) and b[1]['fraction'] is None and b[9]['fraction'] == 0.5
    assert inject.snr_bin([5.0, 5.0], 5.0, 5.0).tolist() == [0, 0]


def test_report():
    inj = [{'round': 0, 'snr': 3.0, 'recovered': True, 'source': {'class_name': 'b'}},
           {'round': 0, 'snr': 90.0, 'recovered': True, 'source': {'class_name': 'b'}},
           {'round': 1, 'snr': 50.0, 'recovered': False, 'source': None}]
    doc = inject.report('m', inj, [{'round': 0}, {'round': 1}], {'snr_range': [3.0, 100.0]})
    assert doc['class_counts'] == {'b': 2} and sum(d['n'] for d in doc['completeness']) == 3
    json.dumps(doc)


# ---------------------------------------------------------------------------------------------- options

def test_config_defaults():
    assert CONFIG['inject_sources'] == 0 and CONFIG['inject_rounds'] == 1
    assert tuple(CONFIG['inject_snr_range']) == (3.0, 100.0) and CONFIG['inject_seed'] == 0


def test_cli(tmp_path):
    run = _run_py()
    w, img = tmp_path / "w.pt", tmp_path / "a.fits"
    w.write_bytes(b"x")
    img.write_bytes(b"SIMPLE")
    base = ['--weights', str(w), '--image', str(img)]
    a = run.parse_args(base)
    assert (a.inject_sources, a.inject_rounds, a.inject_snr_range, a.inject_seed) == (0, 1, '3,100', 0)
    assert run.validate_args(a) == 0
    good = ['--inject_sources', '100', '--inject_rounds', '3', '--inject_snr_range', '5,5', '--inject_seed', '9']
    assert run.validate_args(run.parse_args(base + good)) == 0
    assert run.parse_snr_range('2.5,50') == (2.5, 50.0)
    for bad in (['--inject_sources', '-1'], ['--inject_rounds', '0'], ['--inject_snr_range', '0,10'],
                ['--inject_snr_range', '10,5'], ['--inject_snr_range', '5'], ['--inject_snr_range', '1,2,3'],
                ['--inject_snr_range', 'a,b'], ['--inject_snr_range=-1,5'], ['--inject_snr_range', '1,inf']):
        assert run.validate_args(run.parse_args(base + bad)) == -1, bad


@pytest.mark.parametrize("kw", [dict(inject_sources=-1), dict(inject_rounds=0), dict(inject_snr_range=(0.0, 1.0)),
                                dict(inject_snr_range=(2.0, 1.0)), dict(inject_snr_range=(1.0,))])
def test_sfinder_rejects_bad_options(kw):
    from caesar_yolo_b200.inference import SFinder
    with pytest.raises(ValueError):
        SFinder(_Model(), dict(CONFIG, **kw))


def test_mask_and_estimator_apply_with_injection(caplog):
    """Injection samples the rms map of the save_bkg_maps options, so it is a consumer of the mask and the estimator."""
    from caesar_yolo_b200.inference import SFinder
    caplog.set_level(logging.WARNING)
    sf = SFinder(_Model(), dict(CONFIG, inject_sources=10, bkg_mask_sources=True, bkg_estimator='median'))
    assert sf.bkg_mask_sources is True and sf.bkg_estimator == 'median' and not caplog.records


class _FakeEngine:
    """What SFinder._run_raster needs of the engine for a grey image, on the CPU: no tile, no record."""
    device = torch.device('cpu')

    def begin(self, tiles):
        pass

    def process_tiles(self, *a, **k):
        pass

    def finish(self):
        return torch.zeros(0, dtype=torch.uint8), 0


@pytest.mark.parametrize("n", [0, 16])
def test_png_warns_once_and_writes_no_file(tmp_path, caplog, n):
    from PIL import Image
    from caesar_yolo_b200.inference import SFinder
    path = str(tmp_path / "p.png")
    Image.fromarray(np.arange(48 * 64, dtype=np.uint8).reshape(48, 64)).save(path)
    out = tmp_path / "out"
    out.mkdir()
    kw = {} if n == 0 else dict(inject_sources=n)
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(out), **kw))
    sf.engine = _FakeEngine()
    caplog.set_level(logging.WARNING)
    assert sf.run() == 0
    warned = [r.getMessage() for r in caplog.records if 'injection' in r.getMessage()]
    assert len(warned) == (1 if n else 0)
    assert 'out_p.json' in os.listdir(str(out)) and not any(f.startswith('inject_') for f in os.listdir(str(out)))


def test_foreign_preprocess_fcn_warns(tmp_path, caplog):
    from caesar_yolo_b200.inference import SFinder
    path = str(tmp_path / "f.fits")
    _header_fits(path)
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(tmp_path), inject_sources=4,
                                preprocess_fcn=lambda cube: cube))
    assert sf.set_img_size_params() == 0
    caplog.set_level(logging.WARNING)
    assert sf._inject_beam() is None
    assert len([r for r in caplog.records if 'injection' in r.getMessage()]) == 1
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(tmp_path), inject_sources=4))
    assert sf.set_img_size_params() == 0
    np.testing.assert_array_equal(sf._inject_beam(), fits.beam_cov_pix(sf.fits.header))


def test_library_exports_the_entries():
    from caesar_yolo_b200 import _capi
    for s in ("cy_inject_sources", "cy_inject_restore", "cy_bkg_grid_sample"):
        assert s in _capi.SYMBOLS and hasattr(ops.lib, s)
    assert ops.INJ_DTYPE.itemsize == 32
