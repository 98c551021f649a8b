"""CPU tests of the background-subtracted and S/N maps' host side: the option surface (config default, CLI flag, the
implied bkg / rms maps), the PNG warning, and the map headers (resmap keeps BUNIT, snrmap leaves it out; BKGMASK,
BKGEST and the CRPIX shift as for the bkg / rms maps)."""
import importlib.util
import logging
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, ops
from caesar_yolo_b200.config import CONFIG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_snrmap", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _Model:
    names = {0: 'a'}


def test_config_default():
    assert CONFIG['save_snr_maps'] is False


def test_cli_flag_implies_bkg_maps():
    run = _run_py()
    a = run.parse_args(['--weights', 'w.pt'])
    assert a.save_snr_maps is False and a.save_bkg_maps is False
    a = run.parse_args(['--weights', 'w.pt', '--save_snr_maps', '--bkg_box', '51', '--bkg_grid', '10'])
    assert a.save_snr_maps is True and a.save_bkg_maps is True and (a.bkg_box, a.bkg_grid) == (51, 10)
    assert a.measure_sources is False   # the maps do not imply the per-source measurements
    a = run.parse_args(['--weights', 'w.pt', '--save_bkg_maps'])
    assert a.save_snr_maps is False and a.save_bkg_maps is True


def test_cli_validation_applies_to_the_option(tmp_path):
    run = _run_py()
    w, img = tmp_path / "w.pt", tmp_path / "a.fits"
    w.write_bytes(b"x")
    img.write_bytes(b"SIMPLE")
    base = ['--weights', str(w), '--image', str(img), '--save_snr_maps']
    assert run.validate_args(run.parse_args(base)) == 0
    for bad in (['--bkg_box', '100'], ['--bkg_grid', '0']):
        assert run.validate_args(run.parse_args(base + bad)) == -1, bad


@pytest.mark.parametrize("kw,snr,bkg", [({}, False, False), ({'save_snr_maps': True}, True, True),
                                        ({'save_bkg_maps': True}, False, True),
                                        ({'save_snr_maps': True, 'save_bkg_maps': False}, True, True)])
def test_sfinder_option_implies_bkg_maps(kw, snr, bkg):
    from caesar_yolo_b200.inference import SFinder
    sf = SFinder(_Model(), dict(CONFIG, **kw))
    assert sf.save_snr_maps is snr and sf.save_bkg_maps is bkg
    cfg = dict(CONFIG, **kw)
    if 'save_snr_maps' not in kw:
        del cfg['save_snr_maps']
        assert SFinder(_Model(), cfg).save_snr_maps is False   # a config without the key


def test_mask_and_estimator_apply_with_the_option_alone(caplog):
    """save_snr_maps is a consumer of bkg_mask_sources and bkg_estimator through the bkg / rms maps it implies."""
    from caesar_yolo_b200.inference import SFinder
    caplog.set_level(logging.WARNING)
    sf = SFinder(_Model(), dict(CONFIG, save_snr_maps=True, bkg_mask_sources=True, bkg_estimator='median'))
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


@pytest.mark.parametrize("snr", [False, True])
def test_png_warns_once_and_writes_no_map(tmp_path, caplog, snr):
    from PIL import Image
    from caesar_yolo_b200.inference import SFinder
    path = str(tmp_path / "p.png")
    Image.fromarray(np.arange(48 * 64, dtype=np.uint8).reshape(48, 64)).save(path)
    out = tmp_path / "out"
    out.mkdir()
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(out), save_snr_maps=snr, save_bkg_maps=not snr))
    sf.engine = _FakeEngine()
    caplog.set_level(logging.WARNING)
    assert sf.run() == 0
    warned = [r.getMessage() for r in caplog.records if 'FITS images only' in r.getMessage()]
    assert len(warned) == 1 and (('S/N' in warned[0]) is snr)
    files = os.listdir(str(out))
    assert 'out_p.json' in files and not any(f.endswith('map_p.fits') for f in files)


H = {"BMAJ": 0.0025, "BMIN": 0.002, "BPA": 12.5, "BUNIT": "JY/BEAM", "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN",
     "CRVAL1": 150.0, "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.25, "CDELT1": -0.0004, "CDELT2": 0.0004}


def _cards(hdr):
    return [hdr[k:k + 80].decode() for k in range(0, len(hdr), 80)]


@pytest.mark.parametrize("mask,est", [(False, 'mean'), (True, 'mean'), (False, 'median'), (True, 'median')])
def test_header_without_bunit(mask, est):
    """bunit=False removes the BUNIT card and nothing else."""
    with_unit = fits.map_header(H, 37, 23, 120, 45, bkgmask=mask, bkgest=est)
    assert with_unit == fits.map_header(H, 37, 23, 120, 45, bkgmask=mask, bkgest=est, bunit=True)
    without = fits.map_header(H, 37, 23, 120, 45, bkgmask=mask, bkgest=est, bunit=False)
    assert len(without) % 2880 == 0
    a, b = _cards(with_unit), _cards(without)
    unit = [c for c in a if c.startswith("BUNIT   ")]
    assert len(unit) == 1 and not any(c.startswith("BUNIT   ") for c in b)
    assert [c for c in a if c != unit[0]] + ["%-80s" % ""] == b
    assert any(c.startswith("BKGMASK ") for c in b) is mask
    assert any(c.startswith("BKGEST  ") for c in b) is (est == 'median')
    assert fits.map_header({}, 4, 3, bunit=False) == fits.map_header({}, 4, 3)   # no BUNIT to drop


def test_header_round_trip(tmp_path):
    import torch
    nx, ny, x0, y0 = 9, 5, 120, 45
    rows = torch.from_numpy(np.ones((ny, nx), '>f4').view(np.int32))
    for name, unit in (('res', True), ('snr', False)):
        p = str(tmp_path / (name + ".fits"))
        fits.write_map_rows(p, fits.map_header(H, nx, ny, x0, y0, bkgmask=True, bkgest='median', bunit=unit), rows, 0,
                            nx, ny)
        h = fits.FitsImage(p).header
        assert ('BUNIT' in h) is unit and h.get('BUNIT', 'JY/BEAM') == 'JY/BEAM'
        assert h['BKGMASK'] is True and h['BKGEST'] == 'MEDIAN'
        assert h['CRPIX1'] == H['CRPIX1'] - x0 and h['CRPIX2'] == H['CRPIX2'] - y0
        assert h['BMAJ'] == H['BMAJ'] and h['CTYPE2'] == 'DEC--SIN'


def test_library_exports_the_entry():
    from caesar_yolo_b200 import _capi
    assert "cy_bkg_grid_snr_maps" in _capi.SYMBOLS
    assert hasattr(ops.lib, "cy_bkg_grid_snr_maps")
