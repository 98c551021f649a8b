"""CPU tests of the host side of the reliability estimate (reliability): the option surface (config, CLI, the consumers
of the mask and the estimator, the PNG warning), the tables on hand-made inputs and the JSON document."""
import importlib.util
import json
import logging
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import inject, ops, reliability
from caesar_yolo_b200.config import CONFIG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_reliability", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _Model:
    names = {0: 'a', 1: 'b'}


# ---------------------------------------------------------------------------------------------- options

def test_config_default_is_off():
    assert CONFIG['reliability'] is False


def test_cli_flag_sets_the_config_key(tmp_path, monkeypatch):
    run = _run_py()
    w, img = tmp_path / "w.pt", tmp_path / "a.fits"
    w.write_bytes(b"x")
    img.write_bytes(b"SIMPLE")
    base = ['--weights', str(w), '--image', str(img)]
    assert run.parse_args(base).reliability is False
    assert run.validate_args(run.parse_args(base + ['--reliability'])) == 0
    seen = {}

    class FakeSFinder(object):
        def __init__(self, model, config):
            seen.update(config)

        def run(self):
            return 0

    import caesar_yolo_b200.inference as inf
    import caesar_yolo_b200.model as mdl
    monkeypatch.setattr(inf, 'SFinder', FakeSFinder)
    monkeypatch.setattr(mdl, 'YOLO', lambda *a, **k: _Model())
    keep = dict(CONFIG)
    try:
        assert run.main(base + ['--reliability']) == 0
        assert seen['reliability'] is True
        assert run.main(base) == 0
        assert seen['reliability'] is False
    finally:
        CONFIG.clear()
        CONFIG.update(keep)


def test_mask_and_estimator_apply_with_reliability_alone(caplog):
    """The peak S/N is read from the S/N map of the save_bkg_maps options: reliability is a consumer of the mask and
    the estimator, and they warn without it."""
    from caesar_yolo_b200.inference import SFinder
    caplog.set_level(logging.WARNING)
    sf = SFinder(_Model(), dict(CONFIG, reliability=True, bkg_mask_sources=True, bkg_estimator='median'))
    assert sf.reliability is True and sf.bkg_mask_sources is True and sf.bkg_estimator == 'median'
    assert not caplog.records
    sf = SFinder(_Model(), dict(CONFIG, bkg_mask_sources=True, bkg_estimator='median'))
    assert sf.bkg_mask_sources is False and sf.bkg_estimator == 'mean' and len(caplog.records) == 2


class _FakeEngine:
    """What SFinder._run_raster needs of the engine for a grey image, on the CPU: no tile, no record."""
    device = torch.device('cpu')

    def begin(self, tiles):
        pass

    def process_tiles(self, *a, **k):
        pass

    def finish(self):
        return torch.zeros(0, dtype=torch.uint8), 0


@pytest.mark.parametrize("on", [False, True])
def test_png_warns_once_and_writes_no_file(tmp_path, caplog, on):
    from PIL import Image
    from caesar_yolo_b200.inference import SFinder
    path = str(tmp_path / "p.png")
    Image.fromarray(np.arange(48 * 64, dtype=np.uint8).reshape(48, 64)).save(path)
    out = tmp_path / "out"
    out.mkdir()
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(out), reliability=on))
    sf.engine = _FakeEngine()
    caplog.set_level(logging.WARNING)
    assert sf.run() == 0
    warned = [r.getMessage() for r in caplog.records if 'reliability' in r.getMessage()]
    assert len(warned) == (1 if on else 0)
    assert 'out_p.json' in os.listdir(str(out)) and not any(f.startswith('reliability_') for f in os.listdir(str(out)))


def test_foreign_preprocess_fcn_warns(tmp_path, caplog):
    from caesar_yolo_b200 import synth
    from caesar_yolo_b200.inference import SFinder
    path = str(tmp_path / "f.fits")
    synth.write_fits(path, np.ones((64, 80), np.float32), {})
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(tmp_path), reliability=True,
                                preprocess_fcn=lambda cube: cube))
    assert sf.set_img_size_params() == 0
    caplog.set_level(logging.WARNING)
    assert sf._reliability_on() is False
    assert len([r for r in caplog.records if 'reliability' in r.getMessage()]) == 1
    sf = SFinder(_Model(), dict(CONFIG, image_path=path, outdir=str(tmp_path), reliability=True))
    assert sf.set_img_size_params() == 0 and sf._reliability_on() is True


def test_library_exports_the_entries():
    from caesar_yolo_b200 import _capi
    for s in ("cy_negate_rows", "cy_source_peak_snr"):
        assert s in _capi.SYMBOLS and hasattr(ops.lib, s)


# ---------------------------------------------------------------------------------------------- tables

def test_bin_edges_are_those_of_the_completeness_table():
    for lo, hi in ((3.0, 100.0), (5.0, 5.0), (0.5, 2000.0)):
        t = reliability.tables([], [], [], [], lo, hi, 0.5)
        comp = inject.completeness([], [], lo, hi)
        assert t['bin_edges'] == [d['snr_lo'] for d in comp] + [comp[-1]['snr_hi']]
        assert [(d['snr_lo'], d['snr_hi']) for d in t['snr_bins']] == [(d['snr_lo'], d['snr_hi']) for d in comp]
        assert len(t['snr_bins']) == inject.NBINS == len(t['snr_cumulative'])


def test_counts_on_hand_made_inputs():
    lo, hi = 3.0, 300.0        # edges 3 * 10^(k / 5)
    pos = [3.0, 3.5, 4.7, 30.0, 30.0, 299.0, 300.0, 2.0, 400.0, np.nan, np.nan]
    neg = [3.1, 4.0, 31.0, 31.0, 31.0, 1.0, 1.5, 500.0, np.nan]
    t = reliability.tables(pos, neg, [], [], lo, hi, 0.5)
    b = t['snr_bins']
    assert [d['n_pos'] for d in b] == [3, 0, 0, 0, 0, 2, 0, 0, 0, 2]
    assert [d['n_neg'] for d in b] == [2, 0, 0, 0, 0, 3, 0, 0, 0, 0]
    assert b[0]['reliability'] == pytest.approx(1 - 2 / 3)
    assert b[5]['reliability'] == pytest.approx(-0.5)       # not clipped
    assert b[9]['reliability'] == 1.0 and b[1]['reliability'] is None and b[1]['n_neg'] == 0
    assert t['snr_outside'] == {'below': {'n_pos': 1, 'n_neg': 2}, 'above': {'n_pos': 1, 'n_neg': 1},
                                'nan': {'n_pos': 2, 'n_neg': 1}}
    c = t['snr_cumulative']
    e = t['bin_edges']
    for k in range(inject.NBINS):
        assert c[k]['snr_min'] == e[k]
        assert c[k]['n_pos'] == sum(1 for v in pos if v >= e[k])
        assert c[k]['n_neg'] == sum(1 for v in neg if v >= e[k])
    assert (c[0]['n_pos'], c[0]['n_neg']) == (8, 6)
    assert c[0]['reliability'] == pytest.approx(1 - 6 / 8)


def test_bin_without_positive_detections_is_null():
    t = reliability.tables([], [5.0, 50.0], [], [], 3.0, 100.0, 0.5)
    assert all(d['reliability'] is None for d in t['snr_bins'])
    assert sum(d['n_neg'] for d in t['snr_bins']) == 2


def test_score_thresholds_and_table():
    th = reliability.score_thresholds(0.5)
    assert len(th) == 10 and th[0] == 0.5 and th[5] == pytest.approx(0.75) and th[9] == pytest.approx(0.95)
    assert reliability.score_thresholds(0.7)[1] == 0.7 + 0.3 / 10
    sp = np.array([0.5, 0.55, 0.6, 0.9, 0.96], np.float32)
    sn = np.array([0.5, 0.52, 0.91], np.float32)
    t = reliability.tables([], [], sp, sn, 3.0, 100.0, 0.5)
    s = t['score_cumulative']
    assert [d['score_min'] for d in s] == th
    assert [d['n_pos'] for d in s] == [int((sp.astype(np.float64) >= x).sum()) for x in th]
    assert [d['n_neg'] for d in s] == [int((sn.astype(np.float64) >= x).sum()) for x in th]
    assert s[0]['reliability'] == pytest.approx(1 - 3 / 5)


def _src(boxes, scores, cls):
    s = np.zeros(len(boxes), ops.SRC_DTYPE)
    for k, (b, sc, c) in enumerate(zip(boxes, scores, cls)):
        s[k]['x1'], s[k]['y1'], s[k]['x2'], s[k]['y2'] = b
        s[k]['score'], s[k]['cls'] = sc, c
    return s


def test_report_round_trip(tmp_path):
    cat = _src([(1, 2, 10, 12), (20, 20, 30, 31), (40, 5, 44, 9)], [0.9, 0.6, 0.55], [0, 1, 1])
    neg = _src([(3, 3, 8, 8), (50, 50, 60, 60)], [0.7, 0.51], [1, 1])
    pos_peak = (np.array([12.5, np.nan, 3.25], np.float32), np.array([4, -1, 41]), np.array([7, -1, 6]))
    neg_peak = (np.array([4.5, np.nan], np.float32), np.array([5, -1]), np.array([6, -1]))
    params = {'snr_range': [3.0, 100.0], 'score_thr': 0.5, 'bkg_estimator': 'mean', 'bkg_mask_sources': False,
              'bkg_box': 101, 'bkg_grid': 25}
    doc = reliability.report('m', cat, neg, pos_peak, neg_peak, _Model.names, params, 7)
    p = tmp_path / "r.json"
    with open(str(p), 'w') as f:
        json.dump(doc, f, indent=1)
    back = json.load(open(str(p)))
    assert back == doc
    assert back['image_id'] == 'm' and back['n_tiles_rerun'] == 7
    assert back['n_catalog'] == 3 and back['n_negative'] == 2
    assert back['catalog_snr_peak'] == [12.5, None, 3.25]
    d0, d1 = back['negative_detections']
    assert (d0['x1'], d0['y1'], d0['x2'], d0['y2'], d0['class_name'], d0['score']) == (3, 3, 8, 8, 'b',
                                                                                    float(np.float32(0.7)))
    assert (d0['snr_peak'], d0['peak_x'], d0['peak_y']) == (4.5, 5, 6)
    assert (d1['snr_peak'], d1['peak_x'], d1['peak_y']) == (None, None, None)
    pr = back['params']
    assert pr['snr_range'] == [3.0, 100.0] and pr['score_thr'] == 0.5 and pr['bkg_estimator'] == 'mean'
    assert pr['bkg_mask_sources'] is False and (pr['bkg_box'], pr['bkg_grid']) == (101, 25)
    assert pr['bin_edges'] == reliability.tables([], [], [], [], 3.0, 100.0, 0.5)['bin_edges']
    assert pr['score_thresholds'] == reliability.score_thresholds(0.5)
    for k in ('snr_bins', 'snr_cumulative', 'snr_outside', 'score_cumulative'):
        assert k in back
    assert back['snr_outside']['nan'] == {'n_pos': 1, 'n_neg': 1}
    assert back['class_counts'] == {'catalog': {'a': 1, 'b': 2}, 'negative': {'b': 2}}
    assert back['score_cumulative'][0]['n_pos'] == 3 and back['score_cumulative'][0]['n_neg'] == 2
