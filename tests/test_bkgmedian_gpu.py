"""The median estimator on the GPU (cy_noise_pass_median[_masked], cy_bkg_grid_pass_median[_masked], cy_median_update;
SFinder with bkg_estimator = 'median') against the numpy fp64 restatement test_bkgmedian_cpu.ref_median_clip of the
definition in include/caesar_b200.h.

nbkg and iters are exact and bkg is bit-equal to np.median: the select runs on integer counts, so no rounding enters
it.  rms is compared through its square relative to mean (v - c)^2 + (mean (v - c))^2, the bound of the mean path; the
restatement asserts that no kept pixel lies within 1e-9 relative of a clip bound (the pixel equal to the median is
exempt).  Map pixels are held to the tolerance of test_bkgmap_gpu.py."""
import json
import math
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, ops, synth
from test_bkgmap_gpu import _check_map, _gpu_grid, ref_map
from test_bkgmask_cpu import BLANK, HOLE, VALUE, ref_fill
from test_bkgmask_gpu import _masked, _map_fixture, _crowded_boxes, MAP_X0, MAP_R0, ref_mask
from test_bkgmedian_cpu import ref_median_clip
from test_noise_gpu import _gpu_noise, _noise_boxes, _noise_mosaic, _src

pytestmark = pytest.mark.gpu

F = 16
KEYS = ('bkg', 'rms', 'nbkg', 'iters', 'var_scale')


def _frame_values(img, box, frame, r0, r1):
    ny, nx = img.shape
    x1, y1, x2, y2 = np.asarray(box, np.float64)
    bx0, bx1, by0, by1 = math.ceil(x1), math.floor(x2), math.ceil(y1), math.floor(y2)
    if not (bx0 <= bx1 and by0 <= by1):
        return None
    gx0, gx1 = max(bx0 - frame, 0), min(bx1 + frame, nx - 1)
    gy0, gy1 = max(by0 - frame, r0), min(by1 + frame, r1 - 1)
    if gx0 > gx1 or gy0 > gy1:
        return None
    sub = img[gy0:gy1 + 1, gx0:gx1 + 1].astype(np.float64)
    with np.errstate(invalid='ignore'):
        keep = np.isfinite(sub) & (sub != 0)
    hy0, hy1, hx0, hx1 = max(by0, gy0), min(by1, gy1), max(bx0, gx0), min(bx1, gx1)
    if hy0 <= hy1 and hx0 <= hx1:
        keep[hy0 - gy0:hy1 - gy0 + 1, hx0 - gx0:hx1 - gx0 + 1] = False
    return sub[keep]


def ref_median_noise(img, boxes, frame=F, r0=0, r1=None):
    """Frames as test_noise_gpu.ref_noise (img holds NaN for masked pixels), clipped with ref_median_clip."""
    r1 = img.shape[0] if r1 is None else r1
    R = {k: np.zeros(len(boxes)) for k in KEYS}
    R['bkg'][:] = R['rms'][:] = np.nan
    for i, b in enumerate(np.asarray(boxes, np.float64)):
        v = _frame_values(img, b, frame, r0, r1)
        if v is not None:
            for k, x in ref_median_clip(v).items():
                R[k][i] = x
    return R


def ref_median_nodes(img, box, grid):
    """test_bkgmap_gpu.ref_nodes with the median-centred clipping."""
    H, W = img.shape
    h = box // 2
    xs, ys = ops.bkg_grid_nodes(W, grid), ops.bkg_grid_nodes(H, grid)
    a = img.astype(np.float64)
    with np.errstate(invalid='ignore'):
        a[~np.isfinite(a) | (a == 0)] = np.nan
    R = {k: np.zeros((len(ys), len(xs))) for k in KEYS}
    for j, y in enumerate(ys):
        for i, x in enumerate(xs):
            sub = a[max(y - h, 0):y + h + 1, max(x - h, 0):x + h + 1]
            for k, v in ref_median_clip(sub[~np.isnan(sub)]).items():
                R[k][j, i] = v
    R['xs'], R['ys'] = xs, ys
    return R


def _check(got, R):
    np.testing.assert_array_equal(got['nbkg'], R['nbkg'])
    np.testing.assert_array_equal(got['iters'], R['iters'])
    assert np.all(got['done'] == 1)
    ok = R['nbkg'] > 0
    np.testing.assert_array_equal(np.isnan(got['bkg']), ~ok)
    np.testing.assert_array_equal(np.isnan(got['rms']), ~ok)
    np.testing.assert_array_equal(got['bkg'][ok], R['bkg'][ok])          # bit-equal to np.median
    assert np.all(np.abs(got['rms'][ok] ** 2 - R['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])


def _one(values):
    values = set(values)
    assert len(values) == 1
    return values.pop()


def _run_rounds(ranks, n, world, run_round, state_of):
    """Median passes of every rank: each rank runs round r into its own partials and histogram; the partials are
    concatenated in rank order (the all-gather) and the histograms summed (the all-reduce), and every rank updates its
    own state from them.  Asserts that the ranks agree on the active count.  -> passes."""
    dev = state_of(ranks[0]).device
    sels = [torch.empty((n * ops.SELECT_BYTES,), dtype=torch.uint8, device=dev) for _ in ranks]
    active, passes = n, 0
    while active:
        for rnd in range(ops.SELECT_ROUNDS):
            parts, hists = [], []
            for r, sel in zip(ranks, sels):
                part = torch.zeros((n * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev)
                hist = torch.full((n * ops.SELECT_SLOTS,), -1, dtype=torch.int32, device=dev)   # the pass zeroes it
                run_round(r, sel, rnd, part, hist)
                parts.append(part)
                hists.append(hist)
            allp = torch.cat(parts)
            total = torch.stack(hists).to(torch.int64).sum(0)
            assert int(total.max()) < 2 ** 31
            total = total.to(torch.int32)
            acts = [ops.median_update(allp, world, total, n, state_of(r), sel, rnd) for r, sel in zip(ranks, sels)]
            active = _one(acts) if rnd == ops.SELECT_ROUNDS - 1 else active
            assert rnd == ops.SELECT_ROUNDS - 1 or set(acts) == {None}
        passes += 1
        assert passes <= ops.NOISE_MAX_PASSES
    return passes


def _gpu_noise_median(words, big_endian, ncols, boxes, ranges, dev, frame=F, masked=False):
    """test_noise_gpu._gpu_noise with the median rounds (and each rank's mask of its own rows when masked).  Asserts
    that every rank ends with the same state bytes.  -> (NOISE_DTYPE array, passes)."""
    boxes = np.asarray(boxes, np.float64).reshape(-1, 4)
    src_dev = ops.to_device_bytes(_src(boxes), dev)
    n, world = len(boxes), len(ranges)
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ranks = []
    for r0, r1 in ranges:
        state = torch.empty((n * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
        off = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        units = ops.noise_init(src_dev, n, ncols, r0, r1, frame, state, off)
        mask = ops.source_mask(src_dev, n, ncols, r0, r1) if masked else None
        ranks.append((full[r0:max(r1, r0 + 1)], r0, r1, state, off, units, mask))

    def run_round(r, sel, rnd, part, hist):
        buf, r0, r1, state, off, units, mask = r
        ops.noise_pass_median(buf, ncols, big_endian, r0, ncols, src_dev, n, r0, r1, frame, off, units, state, sel,
                              rnd, part, hist, mask)
    passes = _run_rounds(ranks, n, world, run_round, lambda r: r[3])
    states = [r[3].cpu().numpy().view(ops.NOISE_DTYPE) for r in ranks]
    for s in states[1:]:
        assert s.tobytes() == states[0].tobytes()
    return states[0], passes


def _gpu_grid_median(words, big_endian, box, grid, ranges, dev, X0=0, R0=0, W=None, H=None, boxes=None):
    """test_bkgmap_gpu._gpu_grid with the median rounds; with boxes, test_bkgmask_gpu._gpu_grid_masked's mask, probe
    and fill.  -> (nodes [Ny, Nx], bkg map, rms map, passes, filled)."""
    full = torch.from_numpy(np.ascontiguousarray(words)).to(dev)
    ny_img, nx_img = words.shape
    W = nx_img - X0 if W is None else W
    H = ny_img - R0 if H is None else H
    R1 = R0 + H
    nx, ny = len(ops.bkg_grid_nodes(W, grid)), len(ops.bkg_grid_nodes(H, grid))
    n, world = nx * ny, len(ranges)
    if boxes is not None:
        boxes = np.asarray(boxes, np.float64).reshape(-1, 4)
        src_dev = ops.to_device_bytes(_src(boxes), dev)
    ranks = []
    for r0, r1 in ranges:
        state = torch.empty((n * ops.NOISE_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
        off = torch.empty((ny + 1,), dtype=torch.int64, device=dev)
        units = ops.bkg_grid_init(W, R0, R1, r0, r1, box, grid, state, off)
        mask = None if boxes is None else ops.source_mask(src_dev, len(boxes), nx_img, r0, r1)
        ranks.append((full[r0:max(r1, r0 + 1), X0:], r0, r1, state, off, units, mask))

    def run_round(r, sel, rnd, part, hist):
        buf, r0, r1, state, off, units, mask = r
        ops.bkg_grid_pass_median(buf, nx_img, big_endian, r0, W, R0, R1, r0, r1, box, grid, off, units, state, sel, rnd,
                                 part, hist, mask, nx_img, X0)
    passes = _run_rounds(ranks, n, world, run_round, lambda r: r[3])
    filled = 0
    if boxes is not None:
        probes = [torch.empty_like(r[3]) for r in ranks]
        if _one(ops.bkg_grid_probe_init(r[3], n, p) for r, p in zip(ranks, probes)):
            parts = []
            for (buf, r0, r1, state, off, units, _), p in zip(ranks, probes):
                parts.append(ops.bkg_grid_pass(buf, nx_img, big_endian, r0, W, R0, R1, r0, r1, box, grid, off, units, p,
                                               torch.empty((n * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8,
                                                           device=dev)))
            allp = torch.cat(parts)
            filled = _one(ops.bkg_grid_fill(allp, world, nx, ny, r[3]) for r in ranks)
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


def _check_grid(img, got, bkg, rms, box, grid):
    R = ref_median_nodes(img, box, grid)
    _check(got, R)
    H, W = img.shape
    _check_map(bkg, ref_map(R['bkg'], R['xs'], R['ys'], W, H))
    _check_map(rms, ref_map(R['rms'], R['xs'], R['ys'], W, H))
    return R


def _special(boxes, box):
    return int(np.nonzero((boxes == np.asarray(box, np.float64)).all(1))[0][0])


# ---------------------------------------------------------------------------------------------- sources

@pytest.mark.parametrize("big_endian", [True, False])
def test_noise_parity_with_numpy(cuda_dev, big_endian):
    img = _noise_mosaic(5)
    boxes = _noise_boxes(6)
    ny, nx = img.shape
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    got, passes = _gpu_noise_median(words, big_endian, nx, boxes, [(0, ny)], cuda_dev)
    R = ref_median_noise(img, boxes)
    _check(got, R)
    assert passes == R['iters'].max() + 1
    assert np.any(got['iters'] >= 3) and np.any(got['nbkg'] == 0) and np.any(got['nbkg'] % 2 == 0)
    k = _special(boxes, (320, 1520, 380, 1580))   # constant frame: every key ties
    assert got['bkg'][k] == np.float64(np.float32(0.37)) and got['rms'][k] == 0.0 and got['iters'][k] == 1
    # the mean of the same frames differs: the estimator is in effect
    mean, _ = _gpu_noise(words, big_endian, nx, boxes, [(0, ny)], cuda_dev)
    ok = got['nbkg'] > 0
    assert np.any(mean['bkg'][ok] != got['bkg'][ok])


def _row_case(values):
    """A 1-row image: pixel 0 holds a box, pixels 1.. the values; the frame of width len(values) is the values."""
    v = np.asarray(values, np.float32)
    img = np.concatenate([np.float32([7.0]), v])[None, :]
    return img, [(0, 0, 0, 0)], len(v)


def _select_cases():
    rng = np.random.default_rng(3)
    a = np.float32(1.25)
    b = np.nextafter(a, np.float32(2))                   # keys differ in the last byte only
    wide = [np.float32(-1.5), np.float32(1.5)]           # keys differ in the first byte (the sign)
    return {
        'odd': rng.standard_normal(1001) * 1e-3 + 0.01,
        'even': rng.standard_normal(1000) * 1e-3 + 0.01,
        'one': [0.3],
        'two': [0.3, -0.7],
        'constant': np.full(777, 0.37),
        'quantised': np.round(rng.standard_normal(5000) * 3) + 0.0,          # 0 is masked; heavy ties
        'both_signs': rng.standard_normal(2000) * 1e-3,
        'subnormal_and_large': np.concatenate([np.float32(1e-42) * rng.integers(1, 100, 300),
                                               -np.float32(1e-41) * rng.integers(1, 100, 301),
                                               [3e38, -3e38, 2.5e38], rng.standard_normal(50) * 1e-39]),
        'last_byte': np.concatenate([np.full(50, a), np.full(50, b), rng.uniform(0.5, 1.0, 30),
                                     rng.uniform(1.5, 2.0, 30)]),
        'first_byte': np.concatenate([np.full(40, wide[0]), np.full(40, wide[1]), rng.uniform(-3, -2, 20),
                                      rng.uniform(2, 3, 20)]),
    }


@pytest.mark.parametrize("case", sorted(_select_cases()))
def test_select_cases(cuda_dev, case):
    """Frames and node boxes built to stress the select, for the source kernel and the node kernel alike."""
    v = np.asarray(_select_cases()[case], np.float32)
    img, boxes, frame = _row_case(v)
    got, _ = _gpu_noise_median(img.view(np.int32), False, img.shape[1], boxes, [(0, 1)], cuda_dev, frame=frame)
    R = ref_median_noise(img, boxes, frame)
    _check(got, R)
    if case in ('one', 'two', 'constant', 'last_byte', 'first_byte'):   # no clip removes a value here
        assert got['bkg'][0] == np.median(v.astype(np.float64))
    if case == 'last_byte':
        assert got['bkg'][0] == (float(np.float32(1.25)) + float(np.nextafter(np.float32(1.25), np.float32(2)))) / 2
    if case == 'first_byte':
        assert got['bkg'][0] == 0.0
    # the same values as one node box of the lattice (box larger than the row: every node sees all of it)
    row = img[:, 1:]
    nodes, bkg, rms, _, _ = _gpu_grid_median(row.view(np.int32), False, 2 * row.shape[1] + 1, 10 ** 6, [(0, 1)],
                                             cuda_dev)
    _check_grid(row, nodes, bkg, rms, 2 * row.shape[1] + 1, 10 ** 6)
    np.testing.assert_array_equal(nodes['bkg'], got['bkg'][0])


def test_noise_row_split_invariance(cuda_dev):
    img = _noise_mosaic(7)
    boxes = _noise_boxes(8)
    ny, nx = img.shape
    words = img.astype('>f4').view(np.int32)
    one, p1 = _gpu_noise_median(words, True, nx, boxes, [(0, ny)], cuda_dev)
    R = ref_median_noise(img, boxes)
    _check(one, R)
    for cuts in ([490], [520, 1700]):   # 2 and 3 ranges
        edges = [0] + cuts + [ny]
        got, p = _gpu_noise_median(words, True, nx, boxes, list(zip(edges[:-1], edges[1:])), cuda_dev)
        assert p == p1
        for k in ('bkg', 'nbkg', 'iters', 'done'):
            np.testing.assert_array_equal(got[k], one[k])
        ok = one['nbkg'] > 0
        assert np.all(np.abs(got['rms'][ok] ** 2 - one['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])


def test_noise_masked(cuda_dev):
    img = _noise_mosaic(9)
    boxes = np.concatenate([_crowded_boxes(10), _noise_boxes(11)[:100]])
    ny, nx = img.shape
    words = img.astype('<f4').view(np.int32)
    got, _ = _gpu_noise_median(words, False, nx, boxes, [(0, ny)], cuda_dev, masked=True)
    _check(got, ref_median_noise(_masked(img, boxes), boxes))
    two, _ = _gpu_noise_median(words, False, nx, boxes, [(0, 900), (900, ny)], cuda_dev, masked=True)
    for k in ('bkg', 'nbkg', 'iters'):
        np.testing.assert_array_equal(two[k], got[k])


# ---------------------------------------------------------------------------------------------- maps

def _image(seed, ny=530, nx=610):
    img = synth.make_mosaic(ny, nx, seed=seed, nan_border_frac=0.03)
    img[200:330, 300:440] = np.nan
    img[100, 100:140] = np.inf
    img[105:110, 400] = -np.inf
    img[400:412, 200:230] = 0.0
    return img


@pytest.mark.parametrize("big_endian", [True, False])
def test_maps_parity_with_numpy(cuda_dev, big_endian):
    img = _image(5)
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    got, bkg, rms, passes, _ = _gpu_grid_median(words, big_endian, 51, 20, [(0, img.shape[0])], cuda_dev)
    R = _check_grid(img, got, bkg, rms, 51, 20)
    assert passes == R['iters'].max() + 1 and np.any(R['nbkg'] == 0)


def test_maps_region_offset_and_row_split(cuda_dev):
    img = _image(6)
    words = img.astype('>f4').view(np.int32)
    X0, R0, W, H = 37, 50, 501, 433
    one, b1, r1, p1, _ = _gpu_grid_median(words, True, 51, 20, [(R0, R0 + H)], cuda_dev, X0=X0, R0=R0, W=W, H=H)
    R = _check_grid(img[R0:R0 + H, X0:X0 + W], one, b1, r1, 51, 20)
    for cuts in ([265], [100, 101]):
        edges = [R0] + cuts + [R0 + H]
        got, b, r, p, _ = _gpu_grid_median(words, True, 51, 20, list(zip(edges[:-1], edges[1:])), cuda_dev, X0=X0,
                                           R0=R0, W=W, H=H)
        assert p == p1
        for k in ('bkg', 'nbkg', 'iters'):
            np.testing.assert_array_equal(got[k], one[k])
        ok = one['nbkg'] > 0
        assert np.all(np.abs(got['rms'][ok] ** 2 - one['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])
        _check_map(b, ref_map(R['bkg'], R['xs'], R['ys'], W, H))
        _check_map(r, ref_map(R['rms'], R['xs'], R['ys'], W, H))


@pytest.mark.parametrize("H,W,box,grid", [(1, 200, 11, 7), (150, 1, 11, 7), (60, 80, 21, 100), (40, 45, 301, 10),
                                          (77, 103, 3, 1), (64, 96, 9, 4)])
def test_maps_edge_lattices(cuda_dev, H, W, box, grid):
    rng = np.random.default_rng(H * 1000 + W)
    img = (rng.standard_normal((H, W)) * 1e-3 + 0.01).astype(np.float32)
    img[rng.random((H, W)) < 0.05] = np.nan
    got, bkg, rms, _, _ = _gpu_grid_median(img.view(np.int32), False, box, grid, [(0, H)], cuda_dev)
    _check_grid(img, got, bkg, rms, box, grid)


def test_maps_masked_with_hole_fill(cuda_dev):
    img, boxes = _map_fixture(5)
    words = img.astype('>f4').view(np.int32)
    H, W = img.shape[0] - MAP_R0, img.shape[1] - MAP_X0
    got, bkg, rms, _, filled = _gpu_grid_median(words, True, 51, 20, [(MAP_R0, MAP_R0 + 200), (MAP_R0 + 200,
                                                MAP_R0 + H)], cuda_dev, X0=MAP_X0, R0=MAP_R0, W=W, H=H, boxes=boxes)
    region = img[MAP_R0:, MAP_X0:]
    M = ref_mask(boxes, img.shape[1], MAP_R0, MAP_R0 + H)[:, MAP_X0:]
    R = ref_median_nodes(np.where(M, np.float32(np.nan), region), 51, 20)
    ok = R['nbkg'] > 0
    np.testing.assert_array_equal(got['nbkg'], R['nbkg'])
    np.testing.assert_array_equal(got['iters'], R['iters'])
    np.testing.assert_array_equal(got['bkg'][ok], R['bkg'][ok])
    assert np.all(np.abs(got['rms'][ok] ** 2 - R['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])
    with np.errstate(invalid='ignore'):
        data = np.isfinite(region) & (region != 0)
    h = 25
    has = np.array([[data[max(y - h, 0):y + h + 1, max(x - h, 0):x + h + 1].any() for x in R['xs']] for y in R['ys']])
    cls = np.where(ok, VALUE, np.where(has, HOLE, BLANK))
    assert np.any(cls == HOLE) and np.any(cls == BLANK), "no hole or no blank node: the case would be vacuous"
    fb, fr, want_filled, _ = ref_fill(R['bkg'], R['rms'], cls)
    assert filled == want_filled.sum() > 0
    eb, er, _, _ = ref_fill(np.where(ok, got['bkg'], np.nan), np.where(ok, got['rms'], np.nan), cls)
    np.testing.assert_array_equal(got['bkg'], eb)
    np.testing.assert_array_equal(got['rms'], er)
    _check_map(bkg, ref_map(fb, R['xs'], R['ys'], W, H))
    _check_map(rms, ref_map(fr, R['xs'], R['ys'], W, H))


def test_physics_faint_source_field(cuda_dev):
    """Gaussian noise sigma0 on a pedestal b0 with a dense field of faint Gaussians (peaks 0.5 .. 2 sigma0, below any
    3 sigma clip): their pixels survive the clip and pull the mean up; the median moves less."""
    H, W = 400, 450
    sigma0, b0 = 1e-3, 1e-2
    rng = np.random.default_rng(12)
    img = b0 + sigma0 * rng.standard_normal((H, W))
    yy, xx = np.mgrid[0:H, 0:W]
    for x0, y0, A, s in zip(rng.uniform(0, W, 600), rng.uniform(0, H, 600), rng.uniform(0.5, 2, 600) * sigma0,
                            rng.uniform(1.5, 3, 600)):
        y_a, y_b, x_a, x_b = int(max(y0 - 4 * s, 0)), int(min(y0 + 4 * s + 1, H)), int(max(x0 - 4 * s, 0)), \
            int(min(x0 + 4 * s + 1, W))
        img[y_a:y_b, x_a:x_b] += A * np.exp(-0.5 * ((xx[y_a:y_b, x_a:x_b] - x0) ** 2 + (yy[y_a:y_b, x_a:x_b] - y0) ** 2)
                                            / s ** 2)
    img = img.astype(np.float32)
    words = img.view(np.int32)
    med, bm, rm, _, _ = _gpu_grid_median(words, False, 101, 25, [(0, H)], cuda_dev)
    _check_grid(img, med, bm, rm, 101, 25)
    mean, _, _, _ = _gpu_grid(words, False, 101, 25, [(0, H)], cuda_dev)
    dm, dmean = np.abs(med['bkg'] - b0), np.abs(mean['bkg'] - b0)
    assert np.mean(dm) < np.mean(dmean)
    assert np.mean(dm < dmean) > 0.75


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


def _runs(tmp_path, run, make_cfg, image_id, catalog_name):
    """Median twice, median with the mask, mean and without the key: identical median files, the mean's bytes without
    the key, the BKGEST card on the median maps only; the catalogs check against the restatement."""
    kinds = [('med1', dict(bkg_estimator='median')), ('med2', dict(bkg_estimator='median')),
             ('medmask', dict(bkg_estimator='median', bkg_mask_sources=True)),
             ('mean', dict(bkg_estimator='mean')), ('nokey', {})]
    dirs = {}
    for name, kw in kinds:
        out = tmp_path / name
        out.mkdir()
        assert run(make_cfg(str(out), dict(measure_noise=True, save_bkg_maps=True, **kw))) == 0
        dirs[name] = out
    f = {k: _files(d) for k, d in dirs.items()}
    assert f['med1'] == f['med2'] and f['mean'] == f['nokey'] and sorted(f['med1']) == sorted(f['mean'])
    maps = ['bkgmap_%s.fits' % image_id, 'rmsmap_%s.fits' % image_id]
    for m in maps:
        assert fits.FitsImage(str(dirs['med1'] / m)).header.get('BKGEST') == 'MEDIAN'
        assert fits.FitsImage(str(dirs['medmask'] / m)).header.get('BKGEST') == 'MEDIAN'
        assert 'BKGEST' not in fits.FitsImage(str(dirs['mean'] / m)).header
    assert f['med1'][maps[0]] != f['mean'][maps[0]], "the median changed no map: the case would be vacuous"
    assert f['medmask'][maps[0]] != f['med1'][maps[0]]
    cat = json.load(open(str(dirs['med1'] / catalog_name)))
    return dirs, cat


def _check_catalog_noise(objs, img, r0, r1):
    boxes = [(d['x1'], d['y1'], d['x2'], d['y2']) for d in objs]
    R = ref_median_noise(img, boxes, F, r0, r1)
    assert len(objs) > 0
    for d, i in zip(objs, range(len(objs))):
        assert d['nbkg'] == R['nbkg'][i]
        if R['nbkg'][i] > 0:
            assert d['bkg'] == R['bkg'][i]
            assert abs(d['rms'] ** 2 - R['rms'][i] ** 2) <= 1e-12 * R['var_scale'][i]


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
    sfs = []

    def make(out, kw):
        sfs.append(SFinder(model, _config(path, out, True, preprocess_fcn=pp, **kw)))
        return sfs[-1]
    dirs, cat = _runs(tmp_path, lambda sf: sf.run_parallel(), make, 'm', 'catalog_m.json')
    assert len(cat['sources']) >= 10, "no detections: the test would be vacuous"
    r0, r1 = measure_rows(sfs[0].engine.tiles, 1)[0]
    _check_catalog_noise(cat['sources'], img, r0, r1)


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
    dirs, cat = _runs(tmp_path, lambda sf: sf.run(),
                      lambda out, kw: SFinder(model, _config(path, out, False, preprocess_fcn=pp, image_xmin=x0,
                                                             image_xmax=x1, image_ymin=y0, image_ymax=y1,
                                                             bkg_box=51, bkg_grid=20, **kw)), 'g', 'out_g.json')
    crop = img[y0:y1, x0:x1]
    _check_catalog_noise(cat['objs'], crop, 0, y1 - y0)
    m = fits.FitsImage(str(dirs['med1'] / 'bkgmap_g.fits'))
    R = ref_median_nodes(crop, 51, 20)
    _check_map(m.rows(0, y1 - y0).astype(np.float32), ref_map(R['bkg'], R['xs'], R['ys'], x1 - x0, y1 - y0))


def test_engine_refuses_other_estimators(cuda_dev):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.pipeline import Engine, make_pp_config
    eng = Engine(Wt.make_random_weights('n', 5, seed=0), make_pp_config(enabled=False), device=cuda_dev)
    words = torch.zeros((8, 8), dtype=torch.int32, device=cuda_dev)
    with pytest.raises(ops.CaesarB200Error):
        eng.bkg_maps(words, 8, False, 0, 8, 0, 8, 0, 8, 3, 2, estimator='mode')
    with pytest.raises(ops.CaesarB200Error):
        eng.measure_noise(_src([(2, 2, 3, 3)]), words, 8, False, 0, 8, 0, 8, estimator='biweight')
