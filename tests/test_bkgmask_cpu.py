"""CPU tests of the source mask option's host side: the option surface (config default, CLI flag, the warning when no
consumer is on), the BKGMASK card of the map header, and the numpy restatement of the hole fill of a masked node
lattice (include/caesar_b200.h, cy_bkg_grid_fill) that the GPU tests compare against."""
import importlib.util
import logging
import os

import numpy as np
import pytest

from caesar_yolo_b200 import fits
from caesar_yolo_b200.config import CONFIG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

VALUE, HOLE, BLANK = 0, 1, 2


def ref_fill(bkg, rms, cls):
    """Ring fill of a node lattice.  bkg, rms: [Ny, Nx] fp64; cls: VALUE (finite node), HOLE (nbkg = 0 with data under
    the mask) or BLANK (no data).  Ring k fills every unfilled hole with a VALUE among its 8 neighbours after ring k - 1
    with the mean of their bkg and rms, summed in row-major neighbour order; rings repeat until none fills.  Returns
    (bkg, rms, filled: bool [Ny, Nx], rings that filled a node)."""
    b, r, c = np.array(bkg, np.float64), np.array(rms, np.float64), np.array(cls)
    ny, nx = c.shape
    hole0 = c == HOLE
    rings = 0
    while True:
        nb, nr, nc = b.copy(), r.copy(), c.copy()
        changed = 0
        for j in range(ny):
            for i in range(nx):
                if c[j, i] != HOLE:
                    continue
                sb = sr = 0.0
                k = 0
                for jj in (j - 1, j, j + 1):
                    for ii in (i - 1, i, i + 1):
                        if (jj, ii) != (j, i) and 0 <= jj < ny and 0 <= ii < nx and c[jj, ii] == VALUE:
                            sb += float(b[jj, ii])
                            sr += float(r[jj, ii])
                            k += 1
                if k:
                    nb[j, i], nr[j, i], nc[j, i] = sb / k, sr / k, VALUE
                    changed += 1
        if not changed:
            return b, r, hole0 & (c == VALUE), rings
        b, r, c = nb, nr, nc
        rings += 1


def _run_py():
    spec = importlib.util.spec_from_file_location("cy_run_cli_bkgmask", os.path.join(ROOT, "scripts", "run.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _Model:
    names = {0: 'a'}


def test_config_default_and_cli_flag():
    assert CONFIG['bkg_mask_sources'] is False
    run = _run_py()
    a = run.parse_args(['--weights', 'w.pt'])
    assert a.bkg_mask_sources is False
    a = run.parse_args(['--weights', 'w.pt', '--bkg_mask_sources', '--save_bkg_maps'])
    assert a.bkg_mask_sources is True and a.save_bkg_maps is True
    assert a.measure_sources is False and a.measure_noise is False   # the mask implies no consumer


@pytest.mark.parametrize("consumers,want", [({}, False), ({'measure_noise': True}, True),
                                            ({'save_bkg_maps': True}, True),
                                            ({'measure_sources': True}, False)])
def test_option_needs_a_consumer(caplog, consumers, want):
    """Without measure_noise or save_bkg_maps the option logs one warning and is off."""
    from caesar_yolo_b200.inference import SFinder
    caplog.set_level(logging.WARNING)
    sf = SFinder(_Model(), dict(CONFIG, bkg_mask_sources=True, **consumers))
    assert sf.bkg_mask_sources is want
    warned = [r for r in caplog.records if 'bkg_mask_sources' in r.getMessage()]
    assert len(warned) == (0 if want else 1)
    caplog.clear()
    sf = SFinder(_Model(), dict(CONFIG, **consumers))   # the default: no warning
    assert sf.bkg_mask_sources is False and not caplog.records


def test_bkgmask_card():
    h = {"CTYPE1": "RA---SIN", "CRPIX1": 10.0, "BUNIT": "JY/BEAM"}
    plain, masked = fits.map_header(h, 7, 5), fits.map_header(h, 7, 5, bkgmask=True)
    assert plain == fits.map_header(h, 7, 5, bkgmask=False)
    assert b"BKGMASK" not in plain
    cards = [masked[k:k + 80].decode() for k in range(0, len(masked), 80)]
    card = [c for c in cards if c.startswith("BKGMASK ")]
    assert len(card) == 1 and card[0][10:30] == "%20s" % "T"
    assert cards.index(card[0]) < cards.index("%-80s" % "END")
    # the card only adds: dropping it gives the header without the option
    assert (b"".join(c.encode() for c in cards if not c.startswith("BKGMASK ")) + b" " * 80) == plain


def test_bkgmask_card_round_trip(tmp_path):
    p = str(tmp_path / "m.fits")
    import torch
    fits.write_map_rows(p, fits.map_header({}, 4, 3, bkgmask=True),
                        torch.from_numpy(np.ones((3, 4), '>f4').view(np.int32)), 0, 4, 3)
    m = fits.FitsImage(p)
    assert m.header["BKGMASK"] is True
    np.testing.assert_array_equal(m.rows(0, 3).astype(np.float32), np.ones((3, 4), np.float32))


# ---------------------------------------------------------------------------------------------- ring fill

def test_fill_rings_use_the_previous_ring():
    """A row of holes right of one finite node: ring k fills the k-th hole from the value ring k - 1 gave its left
    neighbour, never from a node filled in the same ring."""
    cls = np.array([[VALUE, HOLE, HOLE, HOLE]])
    bkg = np.array([[2.0, np.nan, np.nan, np.nan]])
    rms = np.array([[0.5, np.nan, np.nan, np.nan]])
    b, r, filled, rings = ref_fill(bkg, rms, cls)
    np.testing.assert_array_equal(b, [[2.0, 2.0, 2.0, 2.0]])
    np.testing.assert_array_equal(r, [[0.5, 0.5, 0.5, 0.5]])
    assert rings == 3 and filled.tolist() == [[False, True, True, True]]
    # two finite nodes feed a hole between them in ring 1; the next ring averages the filled values with the others
    cls = np.array([[VALUE, HOLE, VALUE],
                    [HOLE, HOLE, HOLE]])
    bkg = np.array([[1.0, np.nan, 4.0], [np.nan] * 3])
    b, _, filled, rings = ref_fill(bkg, bkg, cls)
    assert rings == 1   # every hole touches a finite node: one ring
    assert b[0, 1] == 2.5 and b[1, 0] == 1.0 and b[1, 2] == 4.0 and b[1, 1] == 2.5
    assert filled.sum() == 4


def test_fill_blank_nodes_neither_filled_nor_feeding():
    cls = np.array([[BLANK, BLANK, BLANK],
                    [BLANK, HOLE, VALUE],
                    [BLANK, BLANK, BLANK]])
    bkg = np.where(cls == VALUE, 3.0, np.nan)
    bkg[0, 0] = 100.0   # a value on a blank node is never read
    b, r, filled, rings = ref_fill(bkg, bkg * 0.1, cls)
    assert b[1, 1] == 3.0 and r[1, 1] == 3.0 * 0.1 and rings == 1
    assert filled.tolist() == [[False] * 3, [False, True, False], [False] * 3]
    assert np.isnan(b[cls == BLANK][1:]).all() and b[0, 0] == 100.0


def test_fill_isolated_holes_stay_nan():
    """Holes cut off from every finite node by blank nodes stay NaN; the others fill."""
    cls = np.full((5, 6), BLANK)
    cls[0:2, 0:2] = HOLE            # an all-hole island in a blank sea
    cls[3:5, 3:6] = HOLE
    cls[4, 5] = VALUE
    bkg = np.where(cls == VALUE, 7.0, np.nan)
    b, r, filled, _ = ref_fill(bkg, bkg, cls)
    assert np.isnan(b[0:2, 0:2]).all() and not filled[0:2, 0:2].any()
    assert (b[3:5, 3:6] == 7.0).all() and filled[3:5, 3:6].sum() == 5
    # a lattice with no finite node at all: nothing fills
    b, _, filled, rings = ref_fill(np.full((3, 3), np.nan), np.full((3, 3), np.nan), np.full((3, 3), HOLE))
    assert np.isnan(b).all() and not filled.any() and rings == 0


def test_fill_fixed_order_means():
    """The neighbours are summed in row-major order, which fixes the rounding: 1e16 + 1 - 1e16 + 1 gives 0 + 1 = 1 in
    fp64 ((1e16 + 1) rounds to 1e16), where the sum in another order would give 2."""
    cls = np.array([[VALUE, VALUE, VALUE],
                    [VALUE, HOLE, BLANK],
                    [BLANK, BLANK, BLANK]])
    bkg = np.array([[1e16, 1.0, -1e16], [1.0, np.nan, np.nan], [np.nan] * 3])
    b, _, _, _ = ref_fill(bkg, bkg, cls)
    assert b[1, 1] == ((((1e16 + 1.0) + -1e16) + 1.0) / 4) == 0.25
    assert ((1.0 + 1.0) + 1e16 + -1e16) / 4 != b[1, 1]   # the order matters for these values
