"""CPU tests of the local background / noise feature's host side: the six catalog keys derived from the clipped frame
statistics (and their null rules), the writer with and without noise results, and the option surface (config defaults,
CLI flags, argument validation)."""
import importlib.util
import json
import math
import os

import numpy as np
import pytest

from caesar_yolo_b200 import catalog, ops
from caesar_yolo_b200.config import CONFIG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {0: 'spurious', 1: 'compact', 2: 'extended', 3: 'extended-multisland', 4: 'flagged'}


def _sources(n):
    src = np.zeros(n, dtype=ops.SRC_DTYPE)
    src['x1'], src['y1'] = 10.0 * np.arange(n), 5.0
    src['x2'], src['y2'] = src['x1'] + 8.0, 12.0
    src['score'], src['cls'] = 0.75, 1
    return src


def _meas(rows):
    """rows of (npix, sum, peak); the other measurement fields are irrelevant here."""
    m = np.zeros(len(rows), dtype=ops.MEAS_DTYPE)
    for i, (npix, s, peak) in enumerate(rows):
        m[i]['npix'], m[i]['sum'], m[i]['peak'] = npix, s, peak
    return m


def _noise(rows):
    """rows of (bkg, rms, nbkg, iters)."""
    z = np.zeros(len(rows), dtype=ops.NOISE_DTYPE)
    for i, (bkg, rms, nbkg, iters) in enumerate(rows):
        z[i]['bkg'], z[i]['rms'], z[i]['nbkg'], z[i]['iters'], z[i]['done'] = bkg, rms, nbkg, iters, 1
    return z


def test_writer_adds_noise_keys_only_with_noise_results(tmp_path):
    m = _meas([(100, 5.0, 0.5), (49, -1.0, 0.1)])
    z = _noise([(0.01, 0.002, 900, 3), (-0.02, 0.004, 700, 5)])
    plain = catalog.measurement_dicts(m, 20.0)
    noisy = catalog.measurement_dicts(m, 20.0, None, z)
    for a, b in zip(plain, noisy):
        assert set(a) == set(catalog.MEASURE_KEYS)
        assert set(b) == set(catalog.MEASURE_KEYS) | set(catalog.NOISE_KEYS)
        assert {k: b[k] for k in catalog.MEASURE_KEYS} == a          # the 13 keys do not change
    p_plain, p_noisy = str(tmp_path / "a.json"), str(tmp_path / "b.json")
    catalog.write_json({"sources": catalog.sources_to_dicts(_sources(2), NAMES, plain)}, p_plain)
    catalog.write_json({"sources": catalog.sources_to_dicts(_sources(2), NAMES, noisy)}, p_noisy)
    assert not any(k in open(p_plain).read() for k in ('"snr"', '"nbkg"', '"flux_err"'))
    got = json.load(open(p_noisy))['sources']
    assert got[0]['nbkg'] == 900 and got[0]['bkg'] == 0.01 and got[0]['rms'] == 0.002
    assert got[0]['snr'] == pytest.approx((0.5 - 0.01) / 0.002, rel=1e-15)
    assert got[0]['flux_bkgsub'] == pytest.approx((5.0 - 100 * 0.01) / 20.0, rel=1e-15)
    assert got[1]['flux_bkgsub'] == pytest.approx((-1.0 + 49 * 0.02) / 20.0, rel=1e-12)
    # the region file does not change with noise keys
    a, b = str(tmp_path / "a.reg"), str(tmp_path / "b.reg")
    catalog.write_ds9(json.load(open(p_plain))['sources'], a)
    catalog.write_ds9(got, b)
    assert open(a).read() == open(b).read()
    objs = catalog.records_to_objs(_sources(2), NAMES, meas=noisy)
    assert objs[1]['nbkg'] == 700


def test_null_rules():
    m = _meas([(100, 5.0, 0.5), (100, 5.0, 0.5), (0, 0.0, np.nan), (100, 5.0, 0.5)])
    z = _noise([(np.nan, np.nan, 0, 0),          # empty frame: every key but nbkg is null
                (0.25, 0.0, 300, 1),             # constant frame: rms = 0 -> no S/N
                (0.01, 0.002, 400, 2),           # empty box: no peak -> no S/N; flux_bkgsub = 0 - 0 * bkg
                (0.01, 0.002, 400, 2)])
    d = catalog.measurement_dicts(m, 20.0, None, z)
    assert d[0]['nbkg'] == 0 and all(d[0][k] is None for k in ('bkg', 'rms', 'snr', 'flux_bkgsub', 'flux_err'))
    assert d[1]['rms'] == 0.0 and d[1]['bkg'] == 0.25 and d[1]['snr'] is None
    assert d[1]['flux_bkgsub'] == pytest.approx((5.0 - 100 * 0.25) / 20.0) and d[1]['flux_err'] == 0.0
    assert d[2]['snr'] is None and d[2]['flux_bkgsub'] == 0.0 and d[2]['flux_err'] == 0.0
    assert d[3]['snr'] is not None
    # no beam area: no flux_bkgsub, no flux_err; bkg, rms, snr stay
    d = catalog.measurement_dicts(m, None, None, z)
    assert all(x['flux_bkgsub'] is None and x['flux_err'] is None for x in d)
    assert d[3]['bkg'] == 0.01 and d[3]['rms'] == 0.002 and d[3]['snr'] == pytest.approx(245.0)
    assert json.dumps(d).count("NaN") == 0


@pytest.mark.parametrize("npix,A", [(3, 17.5), (12, 17.5), (5000, 17.5), (10 ** 6, 40.0)])
def test_flux_err_regimes(npix, A):
    rms = 0.003
    m = _meas([(npix, 1.0, 0.5)])
    z = _noise([(0.0, rms, 800, 2)])
    got = catalog.measurement_dicts(m, A, None, z)[0]['flux_err']
    assert got == pytest.approx(rms * math.sqrt(npix * min(npix, A)) / A, rel=1e-15)
    if npix < A:      # box smaller than the beam: fully correlated noise, rms * npix / A
        assert got == pytest.approx(rms * npix / A, rel=1e-15)
    else:             # box much larger than the beam: one independent value per beam, rms * sqrt(npix / A)
        assert got == pytest.approx(rms * math.sqrt(npix / A), rel=1e-15)


def test_config_defaults():
    assert CONFIG['measure_noise'] is False and CONFIG['noise_frame'] == 16
    assert CONFIG['measure_sources'] is False


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_noise", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_cli_measure_noise_sets_both_keys():
    run = _run_py()
    a = run.parse_args(['--weights', 'w.pt'])
    assert a.measure_noise is False and a.measure_sources is False and a.noise_frame == 16
    a = run.parse_args(['--weights', 'w.pt', '--measure_sources'])
    assert a.measure_sources is True and a.measure_noise is False
    a = run.parse_args(['--weights', 'w.pt', '--measure_noise', '--noise_frame=24'])
    assert a.measure_noise is True and a.measure_sources is True and a.noise_frame == 24


def test_cli_noise_frame_below_one_is_refused(tmp_path):
    run = _run_py()
    w = tmp_path / "w.pt"
    w.write_bytes(b"x")
    img = tmp_path / "a.fits"
    img.write_bytes(b"SIMPLE")
    base = ['--weights', str(w), '--image', str(img), '--measure_noise']
    assert run.validate_args(run.parse_args(base)) == 0
    assert run.validate_args(run.parse_args(base + ['--noise_frame', '1'])) == 0
    assert run.validate_args(run.parse_args(base + ['--noise_frame', '0'])) == -1
    assert run.validate_args(run.parse_args(base + ['--noise_frame=-3'])) == -1
    assert run.main(base + ['--noise_frame', '0']) == 1
