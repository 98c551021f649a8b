"""CPU tests of the median estimator's host side: the option surface (config default, CLI choices, the refusal of other
values, the warning when no consumer is on), the BKGEST card of the map header, and the numpy restatement of the
median-centred clipping (include/caesar_b200.h, median estimator) that the GPU tests compare against, tied to the
astropy restatement oracle.astro.sigma_clipped_stats."""
import importlib.util
import logging
import math
import os

import numpy as np
import pytest

from caesar_yolo_b200 import fits
from caesar_yolo_b200.config import CONFIG
from oracle import astro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAPPA, MAXITERS = 3.0, 5


def ref_median_clip(v):
    """Median-centred sigma clipping of the unmasked values v (fp64 of float32 pixels) -> dict bkg, rms, nbkg, iters,
    var_scale.  bkg is np.median of the last set; rms sums (v - c), (v - c)^2 about c = the previous median, so its
    square is compared relative to var_scale = mean (v - c)^2 + (mean (v - c))^2.  Asserts that no kept pixel lies
    within 1e-9 relative of a clip bound (the pixel equal to the median sits at the centre and is exempt), so a clip
    decision cannot flip on a reordered fp64 sum."""
    v = np.asarray(v, np.float64)
    lo, hi, c, nprev = -np.inf, np.inf, 0.0, -1
    out = dict(bkg=np.nan, rms=np.nan, nbkg=0, iters=0, var_scale=0.0)
    for k in range(MAXITERS + 1):
        kept = v[(v >= lo) & (v <= hi)]
        m = kept.size
        out['iters'] = k
        if m == 0:
            return dict(out, bkg=np.nan, rms=np.nan, nbkg=0)
        d = kept - c
        s1, s2 = d.sum(), (d * d).sum()
        m1 = s1 / m
        sd = math.sqrt(max(s2 / m - m1 * m1, 0.0))
        med = float(np.median(kept))
        out.update(bkg=med, rms=sd, nbkg=m, var_scale=s2 / m + m1 * m1)
        if (k >= 1 and m == nprev) or k == MAXITERS:
            return out
        for b in (med - KAPPA * sd, med + KAPPA * sd):
            near = (np.abs(kept - b) <= 1e-9 * (abs(med) + KAPPA * sd)) & (kept != med)
            assert not near.any(), ("fixture pixel on a clip bound", k)
        lo, hi, c, nprev = max(lo, med - KAPPA * sd), min(hi, med + KAPPA * sd), med, m
    return out


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_bkgmedian", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _Model:
    names = {0: 'a'}


def test_config_default_and_cli_choices(tmp_path):
    assert CONFIG['bkg_estimator'] == 'mean'
    run = _run_py()
    assert run.parse_args(['--weights', 'w.pt']).bkg_estimator == 'mean'
    a = run.parse_args(['--weights', 'w.pt', '--bkg_estimator', 'median', '--measure_noise'])
    assert a.bkg_estimator == 'median' and a.measure_noise is True
    assert run.parse_args(['--weights', 'w.pt', '--bkg_estimator', 'mean']).bkg_estimator == 'mean'
    for bad in ('mode', 'MEDIAN', 'biweight', ''):
        with pytest.raises(SystemExit):
            run.parse_args(['--weights', 'w.pt', '--bkg_estimator', bad])
    # validate_args refuses a value set past the parser
    img, w = tmp_path / "i.fits", tmp_path / "w.pt"
    img.write_bytes(b"x")
    w.write_bytes(b"x")
    a = run.parse_args(['--weights', str(w), '--image', str(img)])
    assert run.validate_args(a) == 0
    a.bkg_estimator = 'mode'
    assert run.validate_args(a) == -1


@pytest.mark.parametrize("consumers,want", [({}, 'mean'), ({'measure_noise': True}, 'median'),
                                            ({'save_bkg_maps': True}, 'median'),
                                            ({'measure_sources': True}, 'mean')])
def test_option_needs_a_consumer(caplog, consumers, want):
    """Without measure_noise or save_bkg_maps the median logs one warning and changes nothing."""
    from caesar_yolo_b200.inference import SFinder
    caplog.set_level(logging.WARNING)
    sf = SFinder(_Model(), dict(CONFIG, bkg_estimator='median', **consumers))
    assert sf.bkg_estimator == want
    warned = [r for r in caplog.records if 'bkg_estimator' in r.getMessage()]
    assert len(warned) == (0 if want == 'median' else 1)
    caplog.clear()
    for cfg in (dict(CONFIG, **consumers), dict(CONFIG, bkg_estimator='mean', **consumers)):
        sf = SFinder(_Model(), cfg)   # the default and an explicit mean: no warning
        assert sf.bkg_estimator == 'mean' and not caplog.records
    cfg = dict(CONFIG, **consumers)
    del cfg['bkg_estimator']
    assert SFinder(_Model(), cfg).bkg_estimator == 'mean'   # a config without the key


@pytest.mark.parametrize("bad", ['mode', 'Median', None, 3])
def test_sfinder_refuses_other_values(bad):
    from caesar_yolo_b200.inference import SFinder
    with pytest.raises(ValueError):
        SFinder(_Model(), dict(CONFIG, bkg_estimator=bad, measure_noise=True))


def test_bkgest_card():
    h = {"CTYPE1": "RA---SIN", "CRPIX1": 10.0, "BUNIT": "JY/BEAM"}
    plain = fits.map_header(h, 7, 5)
    assert plain == fits.map_header(h, 7, 5, bkgest='mean') and b"BKGEST" not in plain
    for mask in (False, True):
        med = fits.map_header(h, 7, 5, bkgmask=mask, bkgest='median')
        cards = [med[k:k + 80].decode() for k in range(0, len(med), 80)]
        card = [c for c in cards if c.startswith("BKGEST  ")]
        assert len(card) == 1 and card[0][10:20] == "'MEDIAN  '"
        assert cards.index(card[0]) < cards.index("%-80s" % "END")
        # the card only adds
        rest = b"".join(c.encode() for c in cards if not c.startswith("BKGEST  ")) + b" " * 80
        assert rest == fits.map_header(h, 7, 5, bkgmask=mask)


def test_bkgest_card_round_trip(tmp_path):
    import torch
    p = str(tmp_path / "m.fits")
    fits.write_map_rows(p, fits.map_header({}, 4, 3, bkgest='median'),
                        torch.from_numpy(np.ones((3, 4), '>f4').view(np.int32)), 0, 4, 3)
    assert fits.FitsImage(p).header["BKGEST"] == "MEDIAN"


# ---------------------------------------------------------------------------------------------- restatement

def _frames(seed):
    rng = np.random.default_rng(seed)
    yield (rng.standard_normal(5001) * 1e-3 + 0.01).astype(np.float32)           # odd count
    yield (rng.standard_normal(4000) * 1e-3 - 0.002).astype(np.float32)          # even count, both signs
    t = (rng.standard_t(1.5, 3000) * 1e-3 + 2e-3).astype(np.float32)             # heavy tails: several clips
    yield t
    g = (rng.standard_normal(6000) * 1e-3).astype(np.float32)
    g[:300] += 0.05                                                               # a bright neighbour
    yield g
    yield np.round(rng.standard_normal(2000) * 4).astype(np.float32) + 0.5       # integer-quantised, ties


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_restatement_matches_astropy_oracle(seed):
    """The restatement's bkg and rms are astropy's sigma_clipped_stats (median, std) at sigma 3, maxiters 5."""
    for v in _frames(seed):
        R = ref_median_clip(v.astype(np.float64))
        _, med, std = astro.sigma_clipped_stats(v.astype(np.float64), sigma=3, maxiters=5)
        assert R['bkg'] == med
        assert abs(R['rms'] ** 2 - std ** 2) <= 1e-12 * R['var_scale']
        x, _, _, _ = astro._sigma_clip_core(v.astype(np.float64), 3.0, None, None, 5)
        assert R['nbkg'] == x.size


def test_restatement_median_rule():
    """Odd n: the middle value; even n: (x_(n/2-1) + x_(n/2)) / 2 in fp64, which np.median gives."""
    assert ref_median_clip(np.array([3.0], np.float32))['bkg'] == 3.0
    assert ref_median_clip(np.array([1.0, 2.0], np.float32))['bkg'] == 1.5
    R = ref_median_clip(np.array([0.5] * 7, np.float32))
    assert R['bkg'] == 0.5 and R['rms'] == 0.0 and R['iters'] == 1 and R['nbkg'] == 7
    R = ref_median_clip(np.array([], np.float32))
    assert np.isnan(R['bkg']) and R['nbkg'] == 0 and R['iters'] == 0
    a, b = np.float32(1.0), np.nextafter(np.float32(1.0), np.float32(2))
    assert ref_median_clip(np.array([a, b], np.float32))['bkg'] == (float(a) + float(b)) / 2
