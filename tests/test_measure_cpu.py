"""CPU tests of the per-source measurement feature's host side: beam area / flux density from header cards, the SIN and
TAN sky positions against textbook inversions and hand-computed values, the catalog writer with and without
measurements, and the row ranges the ranks measure."""
import json
import math

import numpy as np
import pytest

from caesar_yolo_b200 import catalog, fits, ops, synth
from caesar_yolo_b200.pipeline import measure_rows

FOURLN2 = 4.0 * math.log(2.0)


# ---------------------------------------------------------------------------------------------- beam area / flux

def test_beam_area_cdelt_from_file(tmp_path):
    path = str(tmp_path / "beam.fits")
    synth.write_fits(path, np.zeros((4, 5), np.float32),
                     {"BMAJ": 0.004, "BMIN": 0.002, "CDELT1": -0.0005, "CDELT2": 0.0005})
    h = fits.FitsImage(path).header
    want = math.pi * 0.004 * 0.002 / FOURLN2 / (0.0005 * 0.0005)
    assert fits.beam_area_pix(h) == pytest.approx(want, rel=1e-12)
    meas = np.zeros(1, dtype=ops.MEAS_DTYPE)
    meas['sum'] = 3.5
    d = catalog.measurement_dicts(meas, fits.beam_area_pix(h))[0]
    assert d['flux'] == pytest.approx(3.5 / want, rel=1e-12)


def test_beam_area_cd_matrix_and_pc():
    rho = math.radians(30.0)
    s = 0.0005
    cd = {"CD1_1": -s * math.cos(rho), "CD1_2": s * math.sin(rho), "CD2_1": s * math.sin(rho), "CD2_2": s * math.cos(rho)}
    h = dict(BMAJ=0.003, BMIN=0.003, **cd)
    want = math.pi * 0.003 * 0.003 / FOURLN2 / (s * s)
    assert fits.beam_area_pix(h) == pytest.approx(want, rel=1e-12)
    # PC with CDELT, and CROTA2 with CDELT: the same pixel area
    h_pc = dict(BMAJ=0.003, BMIN=0.003, CDELT1=-s, CDELT2=s, PC1_1=math.cos(rho), PC1_2=-math.sin(rho),
                PC2_1=math.sin(rho), PC2_2=math.cos(rho))
    assert fits.beam_area_pix(h_pc) == pytest.approx(want, rel=1e-12)
    h_rot = dict(BMAJ=0.003, BMIN=0.003, CDELT1=-s, CDELT2=s, CROTA2=30.0)
    assert fits.beam_area_pix(h_rot) == pytest.approx(want, rel=1e-12)
    m = fits.pixel_scale_matrix(h_rot)   # C&G eq. 189: CDELT1 * cos, -CDELT2 * sin / CDELT1 * sin, CDELT2 * cos
    np.testing.assert_allclose(m, [[-s * math.cos(rho), -s * math.sin(rho)], [-s * math.sin(rho), s * math.cos(rho)]])


def test_beam_area_missing_cards_gives_null_flux():
    assert fits.beam_area_pix({"CDELT1": -0.001, "CDELT2": 0.001}) is None            # no beam
    assert fits.beam_area_pix({"BMAJ": 0.004, "BMIN": 0.002}) is None                 # no pixel scale
    assert fits.beam_area_pix({"BMAJ": 0.004, "BMIN": 0.002, "CDELT1": 0.0, "CDELT2": 0.001}) is None
    meas = np.zeros(1, dtype=ops.MEAS_DTYPE)
    meas['sum'] = 1.0
    assert catalog.measurement_dicts(meas, None)[0]['flux'] is None


# ---------------------------------------------------------------------------------------------- SIN / TAN

def _hdr(proj, ra0, dec0, cdelt=0.01, crpix=(101.0, 51.0)):
    return {"CTYPE1": "RA---" + proj, "CTYPE2": "DEC--" + proj, "CRVAL1": ra0, "CRVAL2": dec0, "CRPIX1": crpix[0],
            "CRPIX2": crpix[1], "CDELT1": -cdelt, "CDELT2": cdelt}


def _textbook(proj, h, x, y):
    """Gnomonic / orthographic inversion written directly in standard coordinates (xi, eta) — an independent
    formulation of the same projections."""
    xi = math.radians(h["CDELT1"] * (x + 1 - h["CRPIX1"]))
    eta = math.radians(h["CDELT2"] * (y + 1 - h["CRPIX2"]))
    a0, d0 = math.radians(h["CRVAL1"]), math.radians(h["CRVAL2"])
    if proj == "TAN":
        den = math.cos(d0) - eta * math.sin(d0)
        ra = a0 + math.atan2(xi, den)
        dec = math.atan2(math.sin(d0) + eta * math.cos(d0), math.hypot(xi, den))
    else:
        z = math.sqrt(1.0 - xi * xi - eta * eta)
        ra = a0 + math.atan2(xi, math.cos(d0) * z - eta * math.sin(d0))
        dec = math.asin(eta * math.cos(d0) + math.sin(d0) * z)
    return math.degrees(ra) % 360.0, math.degrees(dec)


def _close_sky(got, want, tol=1e-9):
    dra = (got[0] - want[0] + 180.0) % 360.0 - 180.0
    assert abs(dra) < tol and abs(got[1] - want[1]) < tol, (got, want)


@pytest.mark.parametrize("proj", ["SIN", "TAN"])
def test_crpix_maps_to_crval(proj):
    h = _hdr(proj, 150.25, -33.5)
    ra, dec = fits.pixel_to_world(h, h["CRPIX1"] - 1, h["CRPIX2"] - 1)
    _close_sky((float(ra), float(dec)), (150.25, -33.5), 1e-12)


@pytest.mark.parametrize("proj", ["SIN", "TAN"])
@pytest.mark.parametrize("ra0,dec0,x,y", [(150.25, -33.5, 137.0, 12.0), (45.0, 89.5, 100.0, 150.0),
                                          (0.2, 10.0, 150.0, 60.0), (359.9, -70.0, 20.0, 90.0)])
def test_off_centre_pixels(proj, ra0, dec0, x, y):
    h = _hdr(proj, ra0, dec0)
    ra, dec = fits.pixel_to_world(h, np.array([x]), np.array([y]))
    _close_sky((float(ra[0]), float(dec[0])), _textbook(proj, h, x, y))


@pytest.mark.parametrize("proj", ["SIN", "TAN"])
def test_hand_computed_values(proj):
    # on the equator, 100 pixels east along the row: ra - ra0 = atan(r) (TAN) or asin(r) (SIN), dec = 0
    h = _hdr(proj, 30.0, 0.0)
    r = math.radians(1.0)
    off = math.degrees(math.atan(r) if proj == "TAN" else math.asin(r))
    ra, dec = fits.pixel_to_world(h, h["CRPIX1"] - 1 - 100, h["CRPIX2"] - 1)
    _close_sky((float(ra), float(dec)), (30.0 + off, 0.0), 1e-10)
    # near the pole: 100 pixels north of a reference 0.5 deg from the pole crosses it -> ra0 + 180, dec = 90 - (off - 0.5)
    h = _hdr(proj, 45.0, 89.5)
    ra, dec = fits.pixel_to_world(h, h["CRPIX1"] - 1, h["CRPIX2"] - 1 + 100)
    _close_sky((float(ra), float(dec)), (225.0, 90.0 - (off - 0.5)), 1e-9)
    # crossing RA = 0: 50 pixels east of ra0 = 0.2 on the equator -> 0.2 - 0.5 deg (+360)
    h = _hdr(proj, 0.2, 0.0)
    ra, dec = fits.pixel_to_world(h, h["CRPIX1"] - 1 + 50, h["CRPIX2"] - 1)
    r = math.radians(0.5)
    off = math.degrees(math.atan(r) if proj == "TAN" else math.asin(r))
    _close_sky((float(ra), float(dec)), (360.0 + 0.2 - off, 0.0), 1e-10)
    assert 359.0 < float(ra) < 360.0


@pytest.mark.parametrize("proj", ["SIN", "TAN"])
@pytest.mark.parametrize("x,y", [(100.0, 50.0 - 100), (137.0, 12.0), (70.0, 80.0), (230.0, 51.0)])
def test_field_centred_on_the_pole(proj, x, y):
    # CRVAL2 = 90 and no LONPOLE card: the native longitude of the celestial pole defaults to 0, not 180 (C&G 2002,
    # sect. 2.4: phi_p = 0 when delta_0 >= theta_0 = 90 deg), which turns the field by 180 deg against the
    # limit delta_0 -> 90 of the textbook inversion (that is the LONPOLE = 180 orientation)
    h = _hdr(proj, 45.0, 90.0)
    ra_t, dec_t = _textbook(proj, h, x, y)
    ra, dec = fits.pixel_to_world(h, x, y)
    _close_sky((float(ra), float(dec)), ((ra_t + 180.0) % 360.0, dec_t))
    h["LONPOLE"] = 180.0
    ra, dec = fits.pixel_to_world(h, x, y)
    _close_sky((float(ra), float(dec)), (ra_t, dec_t))
    # hand-computed: 100 pixels below the reference pixel lie on the meridian ra0 + 180 (default) at 90 - atan / asin(r)
    if (x, y) == (100.0, -50.0):
        h.pop("LONPOLE")
        r = math.radians(1.0)
        off = math.degrees(math.atan(r) if proj == "TAN" else math.asin(r))
        ra, dec = fits.pixel_to_world(h, x, y)
        _close_sky((float(ra), float(dec)), (225.0, 90.0 - off), 1e-9)


def test_sin_outside_the_disc_is_nan():
    h = _hdr("SIN", 10.0, 20.0, cdelt=1.0)
    ra, dec = fits.pixel_to_world(h, np.array([h["CRPIX1"] - 1 + 70.0]), np.array([h["CRPIX2"] - 1]))
    assert np.isnan(ra[0]) and np.isnan(dec[0])


@pytest.mark.parametrize("ctypes", [("RA---CAR", "DEC--CAR"), ("GLON-SIN", "GLAT-SIN"), ("DEC--TAN", "RA---TAN"),
                                    ("RA---SIN", "DEC--TAN"), ("", "")])
def test_unsupported_ctype_gives_null(ctypes):
    h = _hdr("SIN", 10.0, 20.0)
    h["CTYPE1"], h["CTYPE2"] = ctypes
    assert fits.pixel_to_world(h, 1.0, 2.0) is None
    meas = np.zeros(1, dtype=ops.MEAS_DTYPE)
    d = catalog.measurement_dicts(meas, None, None)[0]
    assert d['ra'] is None and d['dec'] is None


# ---------------------------------------------------------------------------------------------- catalog writer

NAMES = {0: 'spurious', 1: 'compact', 2: 'extended', 3: 'extended-multisland', 4: 'flagged'}


def _sources():
    src = np.zeros(2, dtype=ops.SRC_DTYPE)
    src[0] = (10.0, 20.0, 30.0, 41.0, 0.875, 1, 1, -1)
    src[1] = (100.0, 5.0, 120.0, 9.0, 0.5, 2, 2, 3)
    return src


# catalog_<id>.json of the two sources above as this build writes it without measurements
PLAIN_JSON = (
    '{\n  "sources": [\n    {\n      "class_id": 1,\n      "class_name": "compact",\n      "edge": true,\n'
    '      "merged": false,\n      "name": "S1",\n      "score": 0.875,\n      "x1": 10.0,\n      "x2": 30.0,\n'
    '      "y1": 20.0,\n      "y2": 41.0\n    },\n    {\n      "class_id": 2,\n      "class_name": "extended",\n'
    '      "edge": 0,\n      "merged": true,\n      "name": "S2",\n      "score": 0.5,\n      "x1": 100.0,\n'
    '      "x2": 120.0,\n      "y1": 5.0,\n      "y2": 9.0\n    }\n  ]\n}')


def test_catalog_without_measurements_unchanged(tmp_path):
    p = str(tmp_path / "c.json")
    catalog.write_json({"sources": catalog.sources_to_dicts(_sources(), NAMES)}, p)
    assert open(p).read() == PLAIN_JSON
    catalog.write_json({"sources": catalog.sources_to_dicts(_sources(), NAMES, None)}, p)
    assert open(p).read() == PLAIN_JSON
    objs = catalog.records_to_objs(_sources(), NAMES)
    assert all(k not in o for o in objs for k in catalog.MEASURE_KEYS)


def test_catalog_with_measurements_nan_is_null(tmp_path):
    meas = np.zeros(2, dtype=ops.MEAS_DTYPE)
    meas[0] = (12, 2.5, 0.75, 15.0, 30.0, 15.25, 30.5, 2.0, 1.0, 45.0)
    meas[1] = (0, 0.0, np.nan, np.nan, np.nan, np.nan, np.nan, np.nan, np.nan, np.nan)
    radec = (np.array([10.5, np.nan]), np.array([-20.25, np.nan]))
    md = catalog.measurement_dicts(meas, 2.0, radec)
    p = str(tmp_path / "c.json")
    catalog.write_json({"sources": catalog.sources_to_dicts(_sources(), NAMES, md)}, p)
    txt = open(p).read()
    assert "NaN" not in txt and "Infinity" not in txt
    got = json.loads(txt)['sources']
    for d in got:
        assert set(catalog.MEASURE_KEYS) <= set(d)
    assert got[0]['npix'] == 12 and got[0]['flux'] == 1.25 and got[0]['ra'] == 10.5 and got[0]['theta'] == 45.0
    assert got[1]['npix'] == 0 and got[1]['sum'] == 0.0
    assert all(got[1][k] is None for k in ('peak', 'peak_x', 'peak_y', 'xc', 'yc', 'a', 'b', 'theta', 'ra', 'dec'))
    assert got[1]['flux'] == 0.0
    objs = catalog.records_to_objs(_sources(), NAMES, meas=md)
    assert objs[0]['xc'] == 15.25 and objs[1]['xc'] is None
    # the region file does not change with measurements
    a, b = str(tmp_path / "a.reg"), str(tmp_path / "b.reg")
    catalog.write_ds9(catalog.sources_to_dicts(_sources(), NAMES), a)
    catalog.write_ds9(json.loads(txt)['sources'], b)
    assert open(a).read() == open(b).read()


# ---------------------------------------------------------------------------------------------- row ownership

@pytest.mark.parametrize("step", [1.0, 0.5, 0.75])
@pytest.mark.parametrize("world", [1, 2, 3, 8, 40])
def test_measure_rows_partition_the_bands(step, world):
    ny = 3000
    tiles = ops.generate_tiles(0, 2047, 0, ny - 1, 512, 512, step, step)
    from caesar_yolo_b200.pipeline import split_tile_rows
    rows = measure_rows(tiles, world)
    parts = split_tile_rows(tiles, world)
    covered = [r for r in rows if r[1] > r[0]]
    assert covered[0][0] == 0 and covered[-1][1] == ny
    for (a0, a1), (b0, b1) in zip(covered, covered[1:]):
        assert a1 == b0                                    # contiguous, in rank order
    for (r0, r1), (a, b) in zip(rows, parts):
        if b > a:
            assert tiles['ymin'][a:b].min() <= r0 and r1 <= tiles['ymax'][a:b].max()   # inside the rank's band
        else:
            assert r0 == r1
