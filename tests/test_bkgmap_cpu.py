"""CPU tests of the background / rms map feature's host side: the option surface (config defaults, CLI flags, argument
validation), the node lattice, the map header (card formats, WCS copied with CRPIX shifted, round trip through
FitsImage and pixel_to_world) and the parallel-by-rows writer on one rank."""
import importlib.util
import os

import numpy as np
import pytest

from caesar_yolo_b200 import fits, ops
from caesar_yolo_b200.config import CONFIG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_bkgmap", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_config_defaults():
    assert CONFIG['save_bkg_maps'] is False and CONFIG['bkg_box'] == 101 and CONFIG['bkg_grid'] == 25


def test_cli_flags():
    run = _run_py()
    a = run.parse_args(['--weights', 'w.pt'])
    assert a.save_bkg_maps is False and a.bkg_box == 101 and a.bkg_grid == 25
    a = run.parse_args(['--weights', 'w.pt', '--save_bkg_maps', '--bkg_box=51', '--bkg_grid', '10'])
    assert a.save_bkg_maps is True and a.bkg_box == 51 and a.bkg_grid == 10
    assert a.measure_sources is False   # the maps do not imply the per-source measurements


def test_cli_box_and_grid_validation(tmp_path):
    run = _run_py()
    w = tmp_path / "w.pt"
    w.write_bytes(b"x")
    img = tmp_path / "a.fits"
    img.write_bytes(b"SIMPLE")
    base = ['--weights', str(w), '--image', str(img), '--save_bkg_maps']
    assert run.validate_args(run.parse_args(base)) == 0
    assert run.validate_args(run.parse_args(base + ['--bkg_box', '3', '--bkg_grid', '1'])) == 0
    for bad in (['--bkg_box', '100'], ['--bkg_box', '1'], ['--bkg_box', '2'], ['--bkg_box=-5'], ['--bkg_grid', '0'],
                ['--bkg_grid=-2']):
        assert run.validate_args(run.parse_args(base + bad)) == -1, bad
    assert run.main(base + ['--bkg_box', '64']) == 1


@pytest.mark.parametrize("n,g,want", [
    (101, 25, [0, 25, 50, 75, 100]),        # W - 1 a multiple of g
    (103, 25, [0, 25, 50, 75, 100, 102]),   # not a multiple: the last step is short
    (26, 25, [0, 25]),
    (1, 25, [0]),                           # one pixel: one node
    (1, 1, [0]),
    (2, 1, [0, 1]),
    (20, 25, [0, 19]),                      # g >= W: the two edges
    (25, 25, [0, 24]),
    (7, 3, [0, 3, 6]),
])
def test_node_lattice(n, g, want):
    assert ops.bkg_grid_nodes(n, g) == want
    assert len(want) == -(-(n - 1) // g) + 1


def test_card_formats():
    assert fits.format_card("CRVAL1", 150.0) == "%-80s" % ("CRVAL1  = %20s" % "150.0")
    assert fits.format_card("CDELT1", -1e-05)[10:30] == "%20s" % "-1.0E-05"
    assert fits.format_card("X", 1.2345e-300)[10:30] == "%20s" % "1.2345E-300"
    assert fits.format_card("X", 3e+20)[10:30] == "%20s" % "3.0E+20"
    assert fits.format_card("NAXIS1", 4096)[10:30] == "%20d" % 4096
    assert fits.format_card("SIMPLE", True)[10:30] == "%20s" % "T"
    assert fits.format_card("CTYPE1", "RA---SIN")[10:20] == "'RA---SIN'"
    assert fits.format_card("BUNIT", "Jy")[10:20] == "'Jy      '"
    assert fits.format_card("OBJECT", "it's")[10:20] == "'it''s   '"
    for v in (0.1, -0.0004, 1 / 3.0, 123456789.123456789, 2.5e-7, -7.77e100):
        c = fits.format_card("V", v)
        assert len(c) == 80 and "e" not in c[10:] and "." in c[10:].split("E")[0]
        assert fits._value(c[10:]) == v
    with pytest.raises(ValueError):
        fits.format_card("V", float("nan"))


WCS = {"BMAJ": 0.0025, "BMIN": 0.002, "BPA": 12.5, "BUNIT": "JY/BEAM", "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN",
       "CRVAL1": 150.0, "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.25, "CUNIT1": "deg", "CUNIT2": "deg",
       "RADESYS": "FK5", "EQUINOX": 2000.0, "LONPOLE": 180.0}
CD = {"CD1_1": -0.0004, "CD1_2": 1.3e-5, "CD2_1": 1.1e-5, "CD2_2": 0.0004}
PC = {"CDELT1": -0.0004, "CDELT2": 0.0004, "PC1_1": 0.99, "PC1_2": -0.05, "PC2_1": 0.05, "PC2_2": 0.99,
      "CROTA2": 0.0}


def _write_map(path, h, nx, ny, x0, y0, data):
    hdr = fits.map_header(h, nx, ny, x0, y0)
    assert len(hdr) % 2880 == 0
    fits.write_map_rows(path, hdr, _rows(data), 0, nx, ny)


def _rows(data):
    import torch
    return torch.from_numpy(np.ascontiguousarray(data, dtype='>f4').view(np.int32))


@pytest.mark.parametrize("scale", [CD, PC], ids=["CD", "PC_CDELT"])
def test_header_round_trip(tmp_path, scale):
    h = dict(WCS, **scale)
    h.update({"NAXIS": 4, "NAXIS3": 1, "CTYPE3": "FREQ", "CRVAL3": 1.4e9, "CTYPE4": "STOKES", "OBJECT": "field"})
    nx, ny, x0, y0 = 37, 23, 120, 45
    data = np.arange(nx * ny, dtype=np.float32).reshape(ny, nx) * np.float32(0.37) - 3
    data[3, 4] = np.nan
    p = str(tmp_path / "m.fits")
    _write_map(p, h, nx, ny, x0, y0, data)
    assert os.path.getsize(p) % 2880 == 0
    m = fits.FitsImage(p)
    assert (m.nx, m.ny, m.bitpix) == (nx, ny, -32) and m.is_raw_f32
    got = m.rows(0, ny).astype(np.float32)
    np.testing.assert_array_equal(got, data)
    for k, v in h.items():
        if k in ("CRPIX1", "CRPIX2"):
            continue
        if k.endswith(("3", "4")) or k in ("NAXIS", "OBJECT"):
            assert k not in m.header or k == "NAXIS"   # only axes 1 and 2 are kept
            continue
        assert m.header[k] == v and type(m.header[k]) is type(v), k
    assert m.header["NAXIS"] == 2
    assert m.header["CRPIX1"] == h["CRPIX1"] - x0 and m.header["CRPIX2"] == h["CRPIX2"] - y0
    i, j = np.meshgrid(np.arange(nx, dtype=np.float64), np.arange(ny, dtype=np.float64))
    ra_m, dec_m = fits.pixel_to_world(m.header, i, j)
    ra_i, dec_i = fits.pixel_to_world(h, i + x0, j + y0)
    np.testing.assert_allclose(ra_m, ra_i, rtol=0, atol=1e-11)
    np.testing.assert_allclose(dec_m, dec_i, rtol=0, atol=1e-11)
    assert fits.beam_area_pix(m.header) == pytest.approx(fits.beam_area_pix(h), rel=1e-15)


def test_header_without_wcs(tmp_path):
    p = str(tmp_path / "m.fits")
    _write_map(p, {"NAXIS": 2, "NAXIS1": 9, "NAXIS2": 9}, 4, 3, 2, 1, np.ones((3, 4), np.float32))
    m = fits.FitsImage(p)
    assert set(m.header) == {"SIMPLE", "BITPIX", "NAXIS", "NAXIS1", "NAXIS2"}


def test_writer_pieces_and_offset(tmp_path):
    """Rows written in pieces and at a row offset land where a one-piece write puts them."""
    nx, ny = 13, 40
    data = np.random.default_rng(1).standard_normal((ny, nx)).astype(np.float32)
    hdr = fits.map_header({}, nx, ny)
    p = str(tmp_path / "a.fits")
    fits.write_map_rows(p, hdr, _rows(data[:17]), 0, nx, ny, piece_bytes=nx * 4 * 3)
    # the second half as a second "rank" on the same file (rank > 0 does not size the file)
    fits.write_map_rows(p, hdr, _rows(data[17:]), 17, nx, ny, rank=1, piece_bytes=nx * 4 * 5)
    np.testing.assert_array_equal(fits.FitsImage(p).rows(0, ny).astype(np.float32), data)
    q = str(tmp_path / "b.fits")
    _write_map(q, {}, nx, ny, 0, 0, data)
    assert open(p, "rb").read() == open(q, "rb").read()


def test_no_map_option_keeps_config_surface():
    """Without the option the SFinder writes no map: its flag is off by default."""
    from caesar_yolo_b200.inference import SFinder

    class M:
        names = {0: 'a'}
    sf = SFinder(M(), dict(CONFIG))
    assert sf.save_bkg_maps is False and sf.bkg_box == 101 and sf.bkg_grid == 25
