"""Source mask on the GPU (cy_source_mask, cy_noise_pass_masked, cy_bkg_grid_pass_masked, cy_bkg_grid_probe_init,
cy_bkg_grid_fill, SFinder with bkg_mask_sources) against numpy fp64 restatements of the definition in
include/caesar_b200.h: M is rasterised in numpy, its pixels are set to NaN, and the restatements of the noise frames
(test_noise_gpu.ref_noise) and the map nodes (test_bkgmap_gpu.ref_nodes / ref_map) run on that image; the holes are then
filled with test_bkgmask_cpu.ref_fill.  Tolerances are those of the noise and map tests."""
import json
import math
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, ops, synth
from test_bkgmap_gpu import _check_map, _gpu_grid, _image, ref_map, ref_nodes
from test_bkgmask_cpu import BLANK, HOLE, VALUE, ref_fill
from test_noise_gpu import _check, _check_catalog, _gpu_noise, _noise_boxes, _noise_mosaic, _src, ref_noise

pytestmark = pytest.mark.gpu

F = 16


def _boxes(boxes):
    return np.asarray(boxes, np.float64).reshape(-1, 4)


def ref_mask(boxes, ncols, r0, r1):
    """bool [r1 - r0, ncols]: pixel (x, y) of rows [r0, r1) lies in the integer box of a source (float32 coordinates,
    as the catalog holds them)."""
    m = np.zeros((r1 - r0, ncols), bool)
    for s in _src(_boxes(boxes)):
        bx0, bx1 = np.ceil(np.float64(s['x1'])), np.floor(np.float64(s['x2']))
        by0, by1 = np.ceil(np.float64(s['y1'])), np.floor(np.float64(s['y2']))
        if not (bx0 <= bx1 and by0 <= by1):
            continue
        xa, xb, ya, yb = max(bx0, 0), min(bx1, ncols - 1), max(by0, r0), min(by1, r1 - 1)
        if xa <= xb and ya <= yb:
            m[int(ya) - r0:int(yb) - r0 + 1, int(xa):int(xb) + 1] = True
    return m


def pack(m):
    """bool [rows, ncols] -> uint32 words [rows, ceil(ncols / 32)]: bit x & 31 of word x >> 5."""
    rows, ncols = m.shape
    w = (ncols + 31) // 32
    p = np.zeros((rows, w * 32), bool)
    p[:, :ncols] = m
    return np.packbits(p, axis=1, bitorder='little').view('<u4').reshape(rows, w)


def _gpu_mask(boxes, ncols, r0, r1, dev):
    b = _boxes(boxes)
    return ops.source_mask(ops.to_device_bytes(_src(b), dev), len(b), ncols, r0, r1)


def _masked(img, boxes, r0=0):
    """img with the pixels of M set to NaN (rows from r0)."""
    out = img.astype(np.float32).copy()
    out[ref_mask(boxes, img.shape[1], r0, r0 + img.shape[0])] = np.nan
    return out


# ---------------------------------------------------------------------------------------------- mask bits

@pytest.mark.parametrize("ncols", [1, 31, 32, 33, 1000])
def test_mask_bits(cuda_dev, ncols):
    rng = np.random.default_rng(ncols)
    nrows = 700
    cx, cy = rng.uniform(-20, ncols + 20, 150), rng.uniform(-20, nrows + 20, 150)
    w, h = rng.uniform(0, min(ncols, 90) + 2, 150), rng.uniform(0, 300, 150)
    rand = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)        # fractional, overlapping
    nan = np.nan
    special = [(nan, 3, 5, 9), (0, nan, 5, 9), (0, 3, nan, 9), (0, 3, 5, nan),   # NaN coordinates: nothing
               (5, 10, 2, 20), (0, 30, 0, 20),                                   # inverted
               (0.2, 40.5, 0.9, 60), (0, 40.2, 3, 40.7),                          # fractional: empty after ceil / floor
               (ncols, 5, ncols + 10, 15), (-10, 5, -1, 15),                      # off the image
               (0, -50, ncols - 1, -1), (0, nrows, 3, nrows + 40),                # outside the rows
               (0, 100, ncols - 1, 150), (0.5, 120.5, ncols / 2, 170.2),          # overlapping full-width boxes
               (-5, 300, ncols + 5, 310), (ncols - 1, 400, ncols - 1, 405)]       # clipped; the last column only
    boxes = np.concatenate([rand, np.asarray(special, np.float64)])
    for r0, r1 in ((0, nrows), (37, 201), (100, 100), (303, 650)):
        got = _gpu_mask(boxes, ncols, r0, r1, cuda_dev).cpu().numpy().view('<u4')
        want = pack(ref_mask(boxes, ncols, r0, r1))
        assert got.shape == want.shape == (r1 - r0, (ncols + 31) // 32)
        np.testing.assert_array_equal(got, want)
        if ncols % 32 and r1 > r0:
            assert not np.any(got[:, -1] >> np.uint32(ncols % 32)), "bits past ncols"
    assert ref_mask(boxes, ncols, 0, nrows)[300:311, :].all()                 # the cases do what they say
    assert not ref_mask(np.asarray(special[:12]), ncols, 0, nrows).any()


def test_mask_long_hull(cuda_dev):
    """A box of thousands of rows spreads over many work units; no source: all zero."""
    boxes = [(3, -100, 4000, 4500), (100.5, 20, 90, 30), (17, 4000, 17, 4400)]
    got = _gpu_mask(boxes, 4100, 10, 4410, cuda_dev).cpu().numpy().view('<u4')
    np.testing.assert_array_equal(got, pack(ref_mask(boxes, 4100, 10, 4410)))
    got = _gpu_mask(np.zeros((0, 4)), 77, 0, 5, cuda_dev).cpu().numpy()
    assert got.shape == (5, 3) and not got.any()


# ---------------------------------------------------------------------------------------------- noise frames

def _gpu_noise_masked(words, big_endian, ncols, boxes, ranges, dev, frame=F):
    """test_noise_gpu._gpu_noise with each rank's mask of its own rows and the masked pass."""
    src_dev = ops.to_device_bytes(_src(boxes), dev)
    n, world = len(boxes), len(ranges)
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ranks = []
    for r0, r1 in ranges:
        state = torch.empty((n * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
        off = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        units = ops.noise_init(src_dev, n, ncols, r0, r1, frame, state, off)
        mask = ops.source_mask(src_dev, n, ncols, r0, r1)
        ranks.append((full[r0:max(r1, r0 + 1)], r0, r1, state, off, units, mask))
    active, passes = n, 0
    while active:
        parts = [ops.noise_pass_masked(buf, ncols, big_endian, r0, ncols, src_dev, n, r0, r1, frame, off, units, state,
                                       torch.empty((n * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev), m)
                 for buf, r0, r1, state, off, units, m in ranks]
        allp = torch.cat(parts)
        acts = {ops.noise_update(allp, world, n, r[3]) for r in ranks}
        assert len(acts) == 1
        active = acts.pop()
        passes += 1
        assert passes <= ops.NOISE_MAX_PASSES
    states = [r[3].cpu().numpy().view(ops.NOISE_DTYPE) for r in ranks]
    for s in states[1:]:
        assert s.tobytes() == states[0].tobytes()
    return states[0], passes


SMALL, COVER = (600, 1200, 604, 1204), (570, 1170, 640, 1240)   # SMALL's whole frame lies inside COVER


def _crowded_boxes(seed):
    """test_noise_gpu's boxes without those larger than 200 x 200 px (their union would mask most of the image), plus
    SMALL and COVER."""
    b = _noise_boxes(seed)
    b = b[(b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1]) < 200 * 200]
    return np.concatenate([b, np.asarray([SMALL, COVER], np.float64)])


def _isolated(boxes, frame, ny, nx):
    """Sources with a non-empty box inside the image whose frame rectangle meets no other box."""
    b0 = np.ceil(boxes[:, :2])
    b1 = np.floor(boxes[:, 2:])
    out = []
    for k in range(len(boxes)):
        if not (np.all(b0[k] <= b1[k]) and np.all(b0[k] >= 0) and b1[k][0] < nx and b1[k][1] < ny):
            continue
        g0, g1 = b0[k] - frame, b1[k] + frame
        meet = np.all(b0 <= b1, 1) & np.all(b0 <= g1, 1) & np.all(b1 >= g0, 1)
        meet[k] = False
        if not meet.any():
            out.append(k)
    return out


@pytest.mark.parametrize("big_endian", [True, False])
def test_masked_noise_parity(cuda_dev, big_endian):
    img = _noise_mosaic(5)
    boxes = _crowded_boxes(6)
    ny, nx = img.shape
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    got, passes = _gpu_noise_masked(words, big_endian, nx, boxes, [(0, ny)], cuda_dev)
    R = ref_noise(_masked(img, boxes), boxes)
    _check(got, R)
    assert passes == R['iters'].max() + 1
    k = len(boxes) - 2                        # SMALL: its frame is covered by its neighbour
    assert got['nbkg'][k] == 0 and np.isnan(got['bkg'][k]) and np.isnan(got['rms'][k])
    plain, _ = _gpu_noise(words, big_endian, nx, boxes, [(0, ny)], cuda_dev)
    assert plain['nbkg'][k] > 0
    assert np.sum(got['nbkg'] < plain['nbkg']) > 20, "the mask removed no neighbour: the case would be vacuous"
    assert np.all(got['nbkg'] <= plain['nbkg'])


def test_masked_noise_isolated_source_unchanged(cuda_dev):
    """A source whose frame touches no other box gets bit-identical bkg / rms with and without the mask."""
    img = _noise_mosaic(9)
    ny, nx = img.shape
    boxes = _crowded_boxes(10)
    words = img.astype('>f4').view(np.int32)
    iso = _isolated(boxes, F, ny, nx)
    assert len(iso) >= 10
    got, _ = _gpu_noise_masked(words, True, nx, boxes, [(0, ny)], cuda_dev)
    plain, _ = _gpu_noise(words, True, nx, boxes, [(0, ny)], cuda_dev)
    assert got[iso].tobytes() == plain[iso].tobytes()


def test_masked_noise_row_split(cuda_dev):
    img = _noise_mosaic(7)
    ny, nx = img.shape
    boxes = _crowded_boxes(8)
    words = img.astype('>f4').view(np.int32)
    one, p1 = _gpu_noise_masked(words, True, nx, boxes, [(0, ny)], cuda_dev)
    R = ref_noise(_masked(img, boxes), boxes)
    _check(one, R)
    for cuts in ([1202], [1190, 1215], [500, 1202, 1800]):    # through SMALL, COVER and the crowded boxes
        edges = [0] + cuts + [ny]
        got, p = _gpu_noise_masked(words, True, nx, boxes, list(zip(edges[:-1], edges[1:])), cuda_dev)
        assert p == p1
        np.testing.assert_array_equal(got['nbkg'], one['nbkg'])
        np.testing.assert_array_equal(got['iters'], one['iters'])
        ok = one['nbkg'] > 0
        assert np.all(np.abs(got['bkg'][ok] - one['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
        assert np.all(np.abs(got['rms'][ok] ** 2 - one['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])


# ---------------------------------------------------------------------------------------------- maps

def _gpu_grid_masked(words, big_endian, boxes, box, grid, ranges, dev, X0=0, R0=0, W=None, H=None):
    """test_bkgmap_gpu._gpu_grid with the source mask: each rank builds the mask of its rows over the image columns
    (region column x = mask column x + X0), runs the masked passes, the probe and the fill.  Asserts that the ranks agree
    on every count and end with the same state.  -> (nodes, bkg map, rms map, passes, filled)."""
    boxes = _boxes(boxes)
    src_dev = ops.to_device_bytes(_src(boxes), dev)
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ny_img, nx_img = words.shape
    W = nx_img - X0 if W is None else W
    H = ny_img - R0 if H is None else H
    R1 = R0 + H
    nx, ny = len(ops.bkg_grid_nodes(W, grid)), len(ops.bkg_grid_nodes(H, grid))
    n, world = nx * ny, len(ranges)
    ranks = []
    for r0, r1 in ranges:
        state = torch.empty((n * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
        off = torch.empty((ny + 1,), dtype=torch.int64, device=dev)
        units = ops.bkg_grid_init(W, R0, R1, r0, r1, box, grid, state, off)
        mask = ops.source_mask(src_dev, len(boxes), nx_img, r0, r1)
        ranks.append((full[r0:max(r1, r0 + 1), X0:], r0, r1, state, off, units, mask))

    def gather(fn):
        return torch.cat([fn(*r, torch.empty((n * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev))
                          for r in ranks])

    def one(values):
        values = set(values)
        assert len(values) == 1
        return values.pop()

    active, passes = n, 0
    while active:
        allp = gather(lambda buf, r0, r1, state, off, units, m, out: ops.bkg_grid_pass_masked(
            buf, nx_img, big_endian, r0, W, R0, R1, r0, r1, box, grid, off, units, state, out, m, nx_img, X0))
        active = one(ops.noise_update(allp, world, n, r[3]) for r in ranks)
        passes += 1
        assert passes <= ops.NOISE_MAX_PASSES
    probes = [torch.empty_like(r[3]) for r in ranks]
    filled = 0
    if one(ops.bkg_grid_probe_init(r[3], n, p) for r, p in zip(ranks, probes)):
        it = iter(probes)
        allp = gather(lambda buf, r0, r1, state, off, units, m, out: ops.bkg_grid_pass(
            buf, nx_img, big_endian, r0, W, R0, R1, r0, r1, box, grid, off, units, next(it), out))
        filled = one(ops.bkg_grid_fill(allp, world, nx, ny, r[3]) for r in ranks)
    states = [r[3].cpu().numpy().view(ops.NOISE_DTYPE) for r in ranks]
    for s in states[1:]:
        assert s.tobytes() == states[0].tobytes()
    bkg, rms = [], []
    for _, r0, r1, state, _, _, _ in ranks:
        b = torch.empty((r1 - r0, W), dtype=torch.int32, device=dev)
        r = torch.empty_like(b)
        ops.bkg_grid_maps(state, W, R0, R1, r0, r1, box, grid, b, r)
        bkg.append(b.cpu().numpy())
        rms.append(r.cpu().numpy())
    dec = [np.concatenate(m).view('>f4').astype(np.float32) for m in (bkg, rms)]
    return states[0].reshape(ny, nx), dec[0], dec[1], passes, filled


def ref_masked_nodes(region, M, box, grid):
    """Restatement of a masked lattice: ref_nodes of the region with M's pixels set to NaN, the node classes (a hole holds
    a data pixel when M is ignored) and the fill.  -> (R, cls, filled bkg, filled rms, filled)."""
    R = ref_nodes(np.where(M, np.float32(np.nan), region), box, grid)
    with np.errstate(invalid='ignore'):
        data = np.isfinite(region) & (region != 0)
    h = box // 2
    has = np.array([[data[max(y - h, 0):y + h + 1, max(x - h, 0):x + h + 1].any() for x in R['xs']] for y in R['ys']])
    cls = np.where(R['nbkg'] > 0, VALUE, np.where(has, HOLE, BLANK))
    fb, fr, filled, _ = ref_fill(R['bkg'], R['rms'], cls)
    return R, cls, fb, fr, filled


def _check_masked(region, M, got, bkg, rms, filled_count, box, grid):
    R, cls, fb, fr, filled = ref_masked_nodes(region, M, box, grid)
    np.testing.assert_array_equal(got['nbkg'], R['nbkg'])
    np.testing.assert_array_equal(got['iters'], R['iters'])
    assert np.all(got['done'] == 1)
    ok = R['nbkg'] > 0
    assert np.all(np.abs(got['bkg'][ok] - R['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
    assert np.all(np.abs(got['rms'][ok] ** 2 - R['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])
    np.testing.assert_array_equal(~ok & ~np.isnan(got['bkg']), filled)
    np.testing.assert_array_equal(np.isnan(got['bkg']), np.isnan(got['rms']))
    assert filled_count == filled.sum()
    # the fill of the GPU's own finite nodes is exact: the same neighbours summed in the same order
    eb, er, _, _ = ref_fill(np.where(ok, got['bkg'], np.nan), np.where(ok, got['rms'], np.nan), cls)
    np.testing.assert_array_equal(got['bkg'], eb)
    np.testing.assert_array_equal(got['rms'], er)
    H, W = region.shape
    _check_map(bkg, ref_map(fb, R['xs'], R['ys'], W, H))
    _check_map(rms, ref_map(fr, R['xs'], R['ys'], W, H))
    return R, cls, filled


MAP_X0, MAP_R0 = 37, 50                        # X0 % 32 != 0
BIG = (60, 300, 230, 470)                      # node boxes (51 px) inside it: holes
BORDER_SRC = (460, 150, 539, 260)              # right next to the NaN border of columns >= 540


def _map_fixture(seed):
    img = _image(seed)
    img[:, 540:] = np.nan                      # a NaN border wider than half a node box: blank nodes
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(0, img.shape[1], 60), rng.uniform(0, img.shape[0], 60)
    w, h = rng.uniform(2, 40, 60), rng.uniform(2, 40, 60)
    crowd = np.floor(np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1))
    return img, np.concatenate([crowd, np.asarray([BIG, BORDER_SRC], np.float64)])


@pytest.mark.parametrize("big_endian", [True, False])
def test_masked_maps_parity(cuda_dev, big_endian):
    img, boxes = _map_fixture(5)
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    ny, nx = img.shape
    got, bkg, rms, passes, nfill = _gpu_grid_masked(words, big_endian, boxes, 51, 20, [(MAP_R0, ny)], cuda_dev,
                                                     X0=MAP_X0, R0=MAP_R0)
    region = img[MAP_R0:, MAP_X0:]
    M = ref_mask(boxes, nx, MAP_R0, ny)[:, MAP_X0:]
    R, cls, filled = _check_masked(region, M, got, bkg, rms, nfill, 51, 20)
    assert passes == R['iters'].max() + 1
    xs, ys = np.asarray(R['xs']) + MAP_X0, np.asarray(R['ys']) + MAP_R0
    # the cases do what they say: holes under BIG and next to the border filled, the border's blank nodes NaN
    under = (xs[None, :] - 25 >= BIG[0]) & (xs[None, :] + 25 <= BIG[2]) & (ys[:, None] - 25 >= BIG[1]) & \
        (ys[:, None] + 25 <= BIG[3])
    assert under.sum() >= 9 and np.all(filled[under])
    border = xs >= 540 + 25
    assert np.all(cls[:, border] == BLANK) and np.all(np.isnan(got['bkg'][:, border]))
    nxt = (ys[:, None] - 25 >= BORDER_SRC[1]) & (ys[:, None] + 25 <= BORDER_SRC[3]) & \
        (xs[None, :] - 25 >= BORDER_SRC[0]) & (xs[None, :] + 25 <= 539)
    assert nxt.sum() >= 2 and np.all(filled[nxt])
    assert np.all(np.isnan(bkg[:, 577 - MAP_X0:]))          # the border stays NaN in the map (blank corners only)
    assert np.isfinite(bkg[BIG[1] - MAP_R0 + 60, BIG[0] - MAP_X0 + 60])


def test_masked_maps_fully_masked_region(cuda_dev):
    """Every node is a hole with no finite node to fill it from: all NaN, nothing filled."""
    rng = np.random.default_rng(3)
    img = (rng.standard_normal((90, 130)) * 1e-3 + 0.01).astype(np.float32)
    got, bkg, rms, _, nfill = _gpu_grid_masked(img.view(np.int32), False, [(-5, -5, 200, 200)], 31, 10, [(0, 90)],
                                               cuda_dev)
    assert nfill == 0 and np.all(got['nbkg'] == 0) and np.all(np.isnan(got['bkg'])) and np.all(np.isnan(got['rms']))
    assert np.all(np.isnan(bkg)) and np.all(np.isnan(rms))


def test_masked_maps_row_split(cuda_dev):
    img, boxes = _map_fixture(7)
    words = img.astype('>f4').view(np.int32)
    ny, nx = img.shape
    one = _gpu_grid_masked(words, True, boxes, 51, 20, [(MAP_R0, ny)], cuda_dev, X0=MAP_X0, R0=MAP_R0)
    region = img[MAP_R0:, MAP_X0:]
    R, _, filled = _check_masked(region, ref_mask(boxes, nx, MAP_R0, ny)[:, MAP_X0:], one[0], one[1], one[2], one[4],
                                 51, 20)
    ok = R['nbkg'] > 0
    for cuts in ([205], [180, 385]):          # through BORDER_SRC, BIG and crowd boxes
        edges = [MAP_R0] + cuts + [ny]
        got, b, r, p, nfill = _gpu_grid_masked(words, True, boxes, 51, 20, list(zip(edges[:-1], edges[1:])), cuda_dev,
                                               X0=MAP_X0, R0=MAP_R0)
        assert p == one[3] and nfill == one[4]
        np.testing.assert_array_equal(got['nbkg'], one[0]['nbkg'])
        np.testing.assert_array_equal(got['iters'], one[0]['iters'])
        np.testing.assert_array_equal(np.isnan(got['bkg']), np.isnan(one[0]['bkg']))
        assert np.all(np.abs(got['bkg'][ok] - one[0]['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
        assert np.all(np.abs(got['rms'][ok] ** 2 - one[0]['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])
        scale = np.nanmax(np.abs(one[0]['bkg'])) + np.nanmax(R['bkg_scale'])
        assert np.all(np.abs(got['bkg'][filled] - one[0]['bkg'][filled]) <= 1e-12 * scale)
        assert np.all(np.abs(got['rms'][filled] - one[0]['rms'][filled]) <= 1e-12 * np.nanmax(one[0]['rms']))


def test_zero_mask_is_the_unmasked_path(cuda_dev):
    """An empty catalog gives an all-zero mask: states and maps byte-identical to the unmasked entries, no fill."""
    img = _image(5)
    words = img.astype('>f4').view(np.int32)
    want = _gpu_grid(words, True, 51, 20, [(0, 265), (265, img.shape[0])], cuda_dev, X0=MAP_X0)
    got = _gpu_grid_masked(words, True, np.zeros((0, 4)), 51, 20, [(0, 265), (265, img.shape[0])], cuda_dev, X0=MAP_X0)
    assert got[0].tobytes() == want[0].tobytes() and got[3] == want[3] and got[4] == 0
    assert np.any(want[0]['nbkg'] == 0)   # all-NaN nodes exist; they are blank, not holes
    assert got[1].tobytes() == want[1].tobytes() and got[2].tobytes() == want[2].tobytes()


# ---------------------------------------------------------------------------------------------- physics

def test_physics_crowded_field(cuda_dev):
    """Gaussian noise sigma0 on a pedestal b0 with a lattice of bright Gaussians (sigma 5 px, boxes of +-4 sigma, 4 px
    apart) and one extended Gaussian (sigma 20 px, box +-4 sigma) larger than a node box.  Without the mask the wings
    of neighbours inside the frames and node boxes bias bkg high; with it every frame, finite node and filled node is
    within 5 sigma0 / sqrt(n) of b0 (n: the node's own count, or the smallest finite count for a filled node) plus the
    wing beyond the boxes (< 0.01 sigma0), and rms within 5 / sqrt(2 n) + 2 % of the clipped-Gaussian value."""
    H = W = 600
    sigma0, b0 = 1e-3, 1e-2
    rng = np.random.default_rng(21)
    img = b0 + sigma0 * rng.standard_normal((H, W))
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    boxes = []
    for x0, y0, A, s in [(60.3 + 45 * i, 60.6 + 45 * j, 30 * sigma0, 5.0) for j in range(6) for i in range(6)] + \
            [(450.2, 449.7, 30 * sigma0, 20.0)]:
        sub = (slice(max(int(y0 - 6 * s), 0), int(y0 + 6 * s) + 1), slice(max(int(x0 - 6 * s), 0), int(x0 + 6 * s) + 1))
        img[sub] += A * np.exp(-0.5 * ((xx[sub] - x0) ** 2 + (yy[sub] - y0) ** 2) / s ** 2)
        boxes.append((math.floor(x0 - 4 * s), math.floor(y0 - 4 * s), math.ceil(x0 + 4 * s), math.ceil(y0 + 4 * s)))
    img = img.astype(np.float32)
    boxes = np.asarray(boxes, np.float64)
    words = img.view(np.int32)
    crowd = np.arange(36)
    # frames
    plain, _ = _gpu_noise(words, False, W, boxes, [(0, H)], cuda_dev)
    got, _ = _gpu_noise_masked(words, False, W, boxes, [(0, H)], cuda_dev)
    _check(got, ref_noise(_masked(img, boxes), boxes))
    z = (plain['bkg'][crowd] - b0) / (sigma0 / np.sqrt(plain['nbkg'][crowd]))
    assert np.mean(z) > 3, "no bias without the mask: the case would be vacuous"
    n = got['nbkg'].astype(np.float64)
    assert np.all(n > 100)
    assert np.all(np.abs(got['bkg'] - b0) <= 5 * sigma0 / np.sqrt(n) + 0.01 * sigma0)
    assert np.all(np.abs(got['rms'] / sigma0 - 0.985) <= 5 / np.sqrt(2 * n) + 0.02)
    # maps
    nodes0, _, _, _ = _gpu_grid(words, False, 101, 25, [(0, H)], cuda_dev)
    nodes, bkg, rms, _, nfill = _gpu_grid_masked(words, False, boxes, 101, 25, [(0, H)], cuda_dev)
    _, cls, filled = _check_masked(img, ref_mask(boxes, W, 0, H), nodes, bkg, rms, nfill, 101, 25)
    assert filled.sum() >= 4 and np.all(cls != BLANK)
    zn = (nodes0['bkg'] - b0) / (sigma0 / np.sqrt(nodes0['nbkg']))
    assert zn.max() > 10, "no biased node without the mask: the case would be vacuous"
    ok = nodes['nbkg'] > 0
    nn = np.where(ok, nodes['nbkg'], nodes['nbkg'][ok].min()).astype(np.float64)
    assert np.all(np.isfinite(nodes['bkg']))
    assert np.all(np.abs(nodes['bkg'] - b0) <= 5 * sigma0 / np.sqrt(nn) + 0.01 * sigma0)
    assert np.all(np.abs(nodes['rms'] / sigma0 - 0.985) <= 5 / np.sqrt(2 * nn) + 0.02)
    assert np.nanmax(np.abs(bkg - b0)) < 0.5 * sigma0


# ---------------------------------------------------------------------------------------------- end to end

WCS_CARDS = {"BMAJ": 0.0025, "BMIN": 0.002, "CTYPE1": "RA---SIN", "CTYPE2": "DEC--SIN", "CRVAL1": 150.0,
             "CRVAL2": -30.0, "CRPIX1": 700.0, "CRPIX2": 500.0, "CDELT1": -0.0004, "CDELT2": 0.0004,
             "BUNIT": "JY/BEAM"}


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


def _runs(tmp_path, run, make_cfg, image_id):
    """Runs: measure_sources only; noise + maps + mask twice; noise + maps with the option False; without the key.
    Checks the file identities and the card; returns (plain catalog, masked catalog, masked dir, unmasked dir)."""
    kinds = [('plain', dict(measure_sources=True)),
             ('mask1', dict(measure_noise=True, save_bkg_maps=True, bkg_mask_sources=True)),
             ('mask2', dict(measure_noise=True, save_bkg_maps=True, bkg_mask_sources=True)),
             ('off', dict(measure_noise=True, save_bkg_maps=True, bkg_mask_sources=False)),
             ('nokey', dict(measure_noise=True, save_bkg_maps=True))]
    dirs, sfs = {}, {}
    for name, kw in kinds:
        out = tmp_path / name
        out.mkdir()
        sf = make_cfg(str(out), kw)
        assert run(sf) == 0
        dirs[name], sfs[name] = out, sf
    f1, f2, off, nokey = (_files(dirs[k]) for k in ('mask1', 'mask2', 'off', 'nokey'))
    assert f1 == f2 and off == nokey and sorted(f1) == sorted(off)
    maps = ['bkgmap_%s.fits' % image_id, 'rmsmap_%s.fits' % image_id]
    for m in maps:
        assert fits.FitsImage(str(dirs['mask1'] / m)).header.get('BKGMASK') is True
        assert 'BKGMASK' not in fits.FitsImage(str(dirs['off'] / m)).header
        assert f1[m] != off[m], "the mask changed no map: the case would be vacuous"
    assert sfs['mask1'].engine.bkg_holes_filled >= 0
    return dirs, sfs


def test_run_parallel_end_to_end(cuda_dev, tmp_path):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    from caesar_yolo_b200.pipeline import measure_rows
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
    dirs, sfs = _runs(tmp_path, lambda sf: sf.run_parallel(),
                      lambda out, kw: SFinder(model, _config(path, out, True, preprocess_fcn=pp, **kw)), 'm')
    plain = json.load(open(str(dirs['plain'] / "catalog_m.json")))['sources']
    masked = json.load(open(str(dirs['mask1'] / "catalog_m.json")))['sources']
    assert len(plain) >= 10, "no detections: the test would be vacuous"
    eng = sfs['mask1'].engine
    r0, r1 = measure_rows(eng.tiles, 1)[0]
    boxes = [(d['x1'], d['y1'], d['x2'], d['y2']) for d in masked]
    imgm = img.copy()
    imgm[r0:r1] = _masked(img[r0:r1], boxes, r0)
    _check_catalog(plain, masked, imgm, WCS_CARDS, r0, r1, F)
    # the map nodes of the run against the restatement over the same mask
    src = np.zeros(len(boxes), dtype=ops.SRC_DTYPE)
    src['x1'], src['y1'], src['x2'], src['y2'] = np.asarray(boxes, np.float32).T
    mask = eng.source_mask_band(src, eng.tiles)
    r0, r1 = measure_rows(eng.tiles, 1)[0]
    for bad in (eng.source_mask(src, img.shape[1] - 5, r0, r1), eng.source_mask(src, img.shape[1], r0 + 1, r1)):
        with pytest.raises(ops.CaesarB200Error):   # 5 columns short of the region, or other rows
            eng.bkg_maps_band(eng.tiles, mask=bad)
        with pytest.raises(ops.CaesarB200Error):
            eng.measure_noise_band(src, eng.tiles, mask=bad)
    nodes, bkg, rms, (X0, R0, Wr, Hr), _ = eng.bkg_maps_band(eng.tiles, mask=mask)
    hdr = len(fits.map_header(WCS_CARDS, Wr, Hr, X0, R0, bkgmask=True))
    raw = open(str(dirs['mask1'] / 'bkgmap_m.fits'), 'rb').read()
    assert raw[hdr:hdr + Wr * Hr * 4] == bkg.cpu().numpy().tobytes()
    region = img[R0:R0 + Hr, X0:X0 + Wr]
    _check_masked(region, ref_mask(boxes, img.shape[1], R0, R0 + Hr)[:, X0:X0 + Wr], nodes,
                  bkg.cpu().numpy().view('>f4').astype(np.float32), rms.cpu().numpy().view('>f4').astype(np.float32),
                  eng.bkg_holes_filled, 101, 25)


def test_run_serial_crop_end_to_end(cuda_dev, tmp_path):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    from caesar_yolo_b200.preprocessing import ZScaleTransformer, MinMaxNormalizer, DataPreprocessor
    img = np.load(os.path.join(os.path.dirname(__file__), "golden", "galaxy0001.npy")).astype(np.float32)
    if img.ndim == 3:
        img = img[..., 0]
    path = str(tmp_path / "g.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(Wt.make_random_weights('n', 5, seed=0, cls_bias=-16.0))
    ny, nx = img.shape
    x0, y0, x1, y1 = nx // 8, ny // 6, nx - nx // 10, ny - ny // 7
    pp = DataPreprocessor([ZScaleTransformer(contrasts=[.25, .25, .25]), MinMaxNormalizer(norm_min=0, norm_max=255.)])
    dirs, sfs = _runs(tmp_path, lambda sf: sf.run(),
                      lambda out, kw: SFinder(model, _config(path, out, False, preprocess_fcn=pp, image_xmin=x0,
                                                             image_xmax=x1, image_ymin=y0, image_ymax=y1,
                                                             bkg_box=51, bkg_grid=20, **kw)), 'g')
    plain = json.load(open(str(dirs['plain'] / "out_g.json")))['objs']
    masked = json.load(open(str(dirs['mask1'] / "out_g.json")))['objs']
    boxes = [(d['x1'], d['y1'], d['x2'], d['y2']) for d in masked]
    crop = img[y0:y1, x0:x1]
    _check_catalog(plain, masked, _masked(crop, boxes), WCS_CARDS, 0, y1 - y0, F)
    m = fits.FitsImage(str(dirs['mask1'] / 'bkgmap_g.fits'))
    R, cls, fb, fr, filled = ref_masked_nodes(crop, ref_mask(boxes, x1 - x0, 0, y1 - y0), 51, 20)
    _check_map(m.rows(0, y1 - y0).astype(np.float32), ref_map(fb, R['xs'], R['ys'], x1 - x0, y1 - y0))
    assert sfs['mask1'].engine.bkg_holes_filled == filled.sum()
