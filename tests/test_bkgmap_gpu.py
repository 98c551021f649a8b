"""Background and rms maps on the GPU (cy_bkg_grid_init / cy_bkg_grid_pass / cy_noise_update / cy_bkg_grid_maps,
SFinder with save_bkg_maps) against a numpy fp64 restatement of the definition in include/caesar_b200.h: node lattice,
sigma clipping of the node boxes and bilinear interpolation with NaN corners dropped.

Node nbkg and iters are exact; bkg is compared relative to |c| + mean |v - c| of its last pass and rms through its square
relative to mean (v - c)^2 + (mean (v - c))^2, as in test_noise_gpu.py (the scales at which a reordered fp64 sum can
differ; the restatement asserts that no kept pixel lies on a clip bound).  Map pixels are within 1 float32 ulp of the
float32-rounded restatement, with the same NaN positions."""
import math
import os

import numpy as np
import pytest
import torch

from caesar_yolo_b200 import fits, ops, synth

pytestmark = pytest.mark.gpu

KAPPA, MAXITERS = 3.0, 5


def _clip(v):
    """Mean-centred sigma clipping of the unmasked values v -> (bkg, rms, nbkg, iters, bkg_scale, var_scale)."""
    lo, hi, c, nprev = -np.inf, np.inf, 0.0, -1
    out = (np.nan, np.nan, 0, 0, 0.0, 0.0)
    for k in range(MAXITERS + 1):
        kept = v[(v >= lo) & (v <= hi)]
        m = kept.size
        if m == 0:
            return out[:3] + (k,) + out[4:]
        d = kept - c
        s1, s2 = d.sum(), (d * d).sum()
        m1 = s1 / m
        mu = c + m1
        sd = math.sqrt(max(s2 / m - m1 * m1, 0.0))
        out = (mu, sd, m, k, abs(c) + np.abs(d).sum() / m, s2 / m + m1 * m1)
        if (k >= 1 and m == nprev) or k == MAXITERS:
            return out
        for b in (mu - KAPPA * sd, mu + KAPPA * sd):
            near = (np.abs(kept - b) <= 1e-9 * (abs(mu) + KAPPA * sd)) & (kept != mu)
            assert not near.any(), "fixture pixel on a clip bound"
        lo, hi, c, nprev = max(lo, mu - KAPPA * sd), min(hi, mu + KAPPA * sd), mu, m
    return out


def ref_nodes(img, box, grid):
    """img: 2-D float32 region (decoded values).  -> dict of [Ny, Nx] arrays and the node positions xs, ys."""
    H, W = img.shape
    h = box // 2
    xs, ys = ops.bkg_grid_nodes(W, grid), ops.bkg_grid_nodes(H, grid)
    a = img.astype(np.float64)
    with np.errstate(invalid='ignore'):
        a[~np.isfinite(a) | (a == 0)] = np.nan
    R = {k: np.zeros((len(ys), len(xs))) for k in ('bkg', 'rms', 'nbkg', 'iters', 'bkg_scale', 'var_scale')}
    for j, y in enumerate(ys):
        for i, x in enumerate(xs):
            sub = a[max(y - h, 0):y + h + 1, max(x - h, 0):x + h + 1]
            r = _clip(sub[~np.isnan(sub)])
            for k, v in zip(('bkg', 'rms', 'nbkg', 'iters', 'bkg_scale', 'var_scale'), r):
                R[k][j, i] = v
    R['xs'], R['ys'] = xs, ys
    return R


def ref_map(vals, xs, ys, W, H):
    """Bilinear map (fp64) of node values [Ny, Nx], NaN corners dropped with the weights renormalised."""
    xs, ys = np.asarray(xs), np.asarray(ys)
    x, y = np.arange(W), np.arange(H)

    def axis(p, nodes):
        n = len(nodes)
        i = np.clip(np.searchsorted(nodes, p, side='right') - 1, 0, max(n - 2, 0))
        i1 = np.minimum(i + 1, n - 1)
        t = np.where(i1 > i, (p - nodes[i]) / np.where(i1 > i, nodes[i1] - nodes[i], 1), 0.0)
        return i, i1, t
    i, i1, t = axis(x, xs)
    j, j1, u = axis(y, ys)
    T, U = t[None, :], u[:, None]
    s = np.zeros((H, W))
    ws = np.zeros((H, W))
    for jj, ii, wgt in ((j, i, (1 - T) * (1 - U)), (j, i1, T * (1 - U)), (j1, i, (1 - T) * U), (j1, i1, T * U)):
        v = vals[jj[:, None], ii[None, :]]
        ok = ~np.isnan(v)
        s += np.where(ok, wgt * np.where(ok, v, 0), 0)
        ws += np.where(ok, wgt, 0)
    with np.errstate(invalid='ignore', divide='ignore'):
        return np.where(ws > 0, s / np.where(ws > 0, ws, 1), np.nan)


def _gpu_grid(words, big_endian, box, grid, ranges, dev, X0=0, R0=0, W=None, H=None):
    """Region: columns [X0, X0 + W), rows [R0, R0 + H) of the word array.  Every range is one rank with its own buffer
    (starting at its first row), state and unit plan; the partials of each pass are concatenated in range order, like
    the all-gather.  Asserts that the ranks agree on the active count and the final state.  -> (nodes [Ny, Nx], bkg map,
    rms map as float32 [H, W], passes)."""
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
        ranks.append((full[r0:max(r1, r0 + 1), X0:], r0, r1, state, off, units))
    active, passes = n, 0
    while active:
        parts = [ops.bkg_grid_pass(buf, nx_img, big_endian, r0, W, R0, R1, r0, r1, box, grid, off, units, state,
                                   torch.empty((n * ops.NOISE_PARTIAL_BYTES,), dtype=torch.uint8, device=dev))
                 for buf, r0, r1, state, off, units in ranks]
        allp = torch.cat(parts)
        acts = {ops.noise_update(allp, world, n, r[3]) for r in ranks}
        assert len(acts) == 1
        active = acts.pop()
        passes += 1
        assert passes <= ops.NOISE_MAX_PASSES
    states = [r[3].cpu().numpy().view(ops.NOISE_DTYPE) for r in ranks]
    for s in states[1:]:
        assert s.tobytes() == states[0].tobytes()
    bkg, rms = [], []
    for _, r0, r1, state, _, _ in ranks:
        b = torch.empty((r1 - r0, W), dtype=torch.int32, device=dev)
        r = torch.empty_like(b)
        ops.bkg_grid_maps(state, W, R0, R1, r0, r1, box, grid, b, r)
        bkg.append(b.cpu().numpy())
        rms.append(r.cpu().numpy())
    dec = [np.concatenate(m).view('>f4').astype(np.float32) for m in (bkg, rms)]
    return states[0].reshape(ny, nx), dec[0], dec[1], passes


def _check_nodes(got, R):
    np.testing.assert_array_equal(got['nbkg'], R['nbkg'])
    np.testing.assert_array_equal(got['iters'], R['iters'])
    assert np.all(got['done'] == 1)
    ok = R['nbkg'] > 0
    np.testing.assert_array_equal(np.isnan(got['bkg']), ~ok)
    np.testing.assert_array_equal(np.isnan(got['rms']), ~ok)
    assert np.all(np.abs(got['bkg'][ok] - R['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
    assert np.all(np.abs(got['rms'][ok] ** 2 - R['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])


def _check_map(got, want64):
    want = want64.astype(np.float32)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.all(np.abs(got[ok].astype(np.float64) - want[ok]) <= np.spacing(np.abs(want[ok])).astype(np.float64))


def _check_all(img, got, bkg, rms, box, grid):
    R = ref_nodes(img, box, grid)
    _check_nodes(got, R)
    H, W = img.shape
    _check_map(bkg, ref_map(R['bkg'], R['xs'], R['ys'], W, H))
    _check_map(rms, ref_map(R['rms'], R['xs'], R['ys'], W, H))
    return R


# ---------------------------------------------------------------------------------------------- fixtures

NY, NX = 530, 610


def _image(seed):
    img = synth.make_mosaic(NY, NX, seed=seed, nan_border_frac=0.03)   # NaN borders as in primary-beam-cut mosaics
    img[200:330, 300:440] = np.nan                                        # all-masked node boxes (box 51)
    img[100, 100:140] = np.inf
    img[105:110, 400] = -np.inf
    img[400:412, 200:230] = 0.0
    return img


@pytest.mark.parametrize("big_endian", [True, False])
@pytest.mark.parametrize("box,grid", [(51, 20), (101, 25)])
def test_parity_with_numpy(cuda_dev, big_endian, box, grid):
    img = _image(5)
    words = (img.astype('>f4') if big_endian else img.astype('<f4')).view(np.int32)
    got, bkg, rms, passes = _gpu_grid(words, big_endian, box, grid, [(0, NY)], cuda_dev)
    R = _check_all(img, got, bkg, rms, box, grid)
    assert passes == R['iters'].max() + 1
    if box == 51:   # the cases do what they say
        assert np.any(R['nbkg'] == 0), "no all-masked node"
        j, i = np.argwhere(R['nbkg'] == 0)[0]   # the first all-masked node in row-major order
        y, x = R['ys'][j], R['xs'][i]
        # the pixel left of it has the NaN node and a finite one as corners: finite, its weights renormalised
        assert R['nbkg'][j, i - 1] > 0 and np.isnan(bkg[y, x]) and np.isfinite(bkg[y, x - 1])


def test_region_offset(cuda_dev):
    """Columns from X0 and rows from R0: the lattice starts at the region's corner."""
    img = _image(6)
    words = img.astype('>f4').view(np.int32)
    X0, R0, W, H = 37, 50, 501, 433
    got, bkg, rms, _ = _gpu_grid(words, True, 51, 20, [(R0, R0 + H)], cuda_dev, X0=X0, R0=R0, W=W, H=H)
    _check_all(img[R0:R0 + H, X0:X0 + W], got, bkg, rms, 51, 20)


def test_constant_image(cuda_dev):
    img = np.full((90, 130), 0.375, np.float32)   # a binary fraction: every sum of the statistic is exact
    got, bkg, rms, passes = _gpu_grid(img.view(np.int32), False, 31, 10, [(0, 90)], cuda_dev)
    _check_all(img, got, bkg, rms, 31, 10)
    assert np.all(got['rms'] == 0) and np.all(got['bkg'] == 0.375) and np.all(got['iters'] == 1)
    assert np.all(bkg == np.float32(0.375)) and np.all(rms == 0) and passes == 2


@pytest.mark.parametrize("H,W,box,grid", [
    (1, 200, 11, 7),       # one row: one node row
    (150, 1, 11, 7),       # one column
    (60, 80, 21, 100),     # grid >= W and H: nodes on the corners only
    (40, 45, 301, 10),     # box larger than the image: every node sees the whole image
    (77, 103, 3, 1),       # a node per pixel, 3x3 boxes
    (64, 96, 9, 4),
])
def test_edge_lattices(cuda_dev, H, W, box, grid):
    rng = np.random.default_rng(H * 1000 + W)
    img = (rng.standard_normal((H, W)) * 1e-3 + 0.01).astype(np.float32)
    img[rng.random((H, W)) < 0.05] = np.nan
    got, bkg, rms, _ = _gpu_grid(img.view(np.int32), False, box, grid, [(0, H)], cuda_dev)
    _check_all(img, got, bkg, rms, box, grid)


def test_row_split_invariance(cuda_dev):
    img = _image(7)
    words = img.astype('>f4').view(np.int32)
    one, b1, r1, p1 = _gpu_grid(words, True, 101, 25, [(0, NY)], cuda_dev)
    R = _check_all(img, one, b1, r1, 101, 25)
    for cuts in ([265], [100, 101], [13, 300], [0, 529]):
        edges = [0] + cuts + [NY]
        got, b, r, p = _gpu_grid(words, True, 101, 25, list(zip(edges[:-1], edges[1:])), cuda_dev)
        assert p == p1
        np.testing.assert_array_equal(got['nbkg'], one['nbkg'])
        np.testing.assert_array_equal(got['iters'], one['iters'])
        ok = one['nbkg'] > 0
        assert np.all(np.abs(got['bkg'][ok] - one['bkg'][ok]) <= 1e-12 * R['bkg_scale'][ok])
        assert np.all(np.abs(got['rms'][ok] ** 2 - one['rms'][ok] ** 2) <= 1e-12 * R['var_scale'][ok])
        _check_map(b, ref_map(R['bkg'], R['xs'], R['ys'], NX, NY))
        _check_map(r, ref_map(R['rms'], R['xs'], R['ys'], NX, NY))


def test_physics_pedestal_and_noise(cuda_dev):
    """Gaussian noise sigma0 on a pedestal b0 with one bright Gaussian source (peak 1000 sigma0, sigma s px).  Clipping
    removes the source's core; the wings below 3 sigma0 stay and carry at most 2 pi s^2 * 3 sigma0 of flux (the integral
    of a 2-D Gaussian over where it is below a level L is 2 pi s^2 L), so a node's bkg is within 5 sigma0 / sqrt(n) of
    b0 plus that flux over n.  Its rms is within 5 / sqrt(2 n) relative of the clipped-Gaussian value (a Gaussian clipped
    at +-3 sigma converges to a std ~1.5 % below sigma0) plus the wing flux's share of the variance."""
    H, W, s = 400, 450, 3.0
    sigma0, b0 = 1e-3, 1e-2
    rng = np.random.default_rng(11)
    img = b0 + sigma0 * rng.standard_normal((H, W))
    yy, xx = np.mgrid[0:H, 0:W]
    img += 1000 * sigma0 * np.exp(-0.5 * ((xx - 201.3) ** 2 + (yy - 187.6) ** 2) / s ** 2)
    img = img.astype(np.float32)
    got, bkg, rms, _ = _gpu_grid(img.view(np.int32), False, 101, 25, [(0, H)], cuda_dev)
    _check_all(img, got, bkg, rms, 101, 25)
    n = got['nbkg'].astype(np.float64)
    wing = 2 * math.pi * s * s * 3 * sigma0
    assert np.all(np.abs(got['bkg'] - b0) <= 5 * sigma0 / np.sqrt(n) + wing / n)
    assert np.all(np.abs(got['rms'] / sigma0 - 0.985) <= 5 / np.sqrt(2 * n) + 0.01 + 3 * wing / n / sigma0)
    assert np.nanmax(np.abs(bkg - b0)) < 0.5 * sigma0   # the map interpolates nodes that each pass the bound above


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


def _map_files(outdir, image_id):
    return [os.path.join(outdir, p + image_id + '.fits') for p in ('bkgmap_', 'rmsmap_')]


def _same_outputs_plus_maps(plain, maps, image_id):
    """A run without the option writes no map; with it, the same files byte for byte plus the two maps."""
    names = sorted(os.listdir(str(plain)))
    assert names and not any(os.path.basename(p) in names for p in _map_files('', image_id))
    assert sorted(os.listdir(str(maps))) == sorted(names + [os.path.basename(p) for p in _map_files('', image_id)])
    for f in names:
        assert open(str(plain / f), 'rb').read() == open(str(maps / f), 'rb').read(), f


def _check_files(outdir, image_id, W, H, X0, R0, bkg_dev, rms_dev):
    hdr_len = len(fits.map_header(WCS_CARDS, W, H, X0, R0))
    for path, want in zip(_map_files(outdir, image_id), (bkg_dev, rms_dev)):
        m = fits.FitsImage(path)
        assert (m.nx, m.ny) == (W, H)
        assert m.header['CRPIX1'] == WCS_CARDS['CRPIX1'] - X0 and m.header['CRPIX2'] == WCS_CARDS['CRPIX2'] - R0
        assert m.header['BUNIT'] == 'JY/BEAM' and m.header['CTYPE1'] == 'RA---SIN'
        raw = open(path, 'rb').read()
        assert len(raw) % 2880 == 0 and m.offset == hdr_len
        assert raw[hdr_len:hdr_len + W * H * 4] == want.cpu().numpy().tobytes()
        assert raw[hdr_len + W * H * 4:] == b'\0' * (len(raw) - hdr_len - W * H * 4)


def test_run_serial_crop_end_to_end(cuda_dev, tmp_path):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    img = synth.make_mosaic(700, 900, seed=4, nan_border_frac=0.02)
    path = str(tmp_path / "g.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(Wt.make_random_weights('n', 5, seed=0, cls_bias=-16.0))
    x0, y0, x1, y1 = 113, 87, 811, 640
    outs = []
    for k, maps in enumerate((False, True, True)):
        out = tmp_path / ("out%d" % k)
        out.mkdir()
        sf = SFinder(model, _config(path, str(out), False, image_xmin=x0, image_xmax=x1, image_ymin=y0, image_ymax=y1,
                                    save_bkg_maps=maps, bkg_box=51, bkg_grid=20))
        assert sf.run() == 0
        outs.append(out)
    _same_outputs_plus_maps(outs[0], outs[1], 'g')
    dev_img = torch.from_numpy(img[y0:y1].astype('>f4').view(np.int32)).to(cuda_dev)
    nodes, bkg, rms = sf.engine.bkg_maps(dev_img[:, x0:], img.shape[1], True, 0, x1 - x0, 0, y1 - y0, 0, y1 - y0,
                                         51, 20)
    _check_files(str(outs[1]), 'g', x1 - x0, y1 - y0, x0, y0, bkg, rms)
    for a, b in zip(_map_files(str(outs[1]), 'g'), _map_files(str(outs[2]), 'g')):
        assert open(a, 'rb').read() == open(b, 'rb').read()
    crop = img[y0:y1, x0:x1]
    R = ref_nodes(crop, 51, 20)
    _check_nodes(nodes, R)
    _check_map(fits.FitsImage(_map_files(str(outs[1]), 'g')[0]).rows(0, y1 - y0).astype(np.float32),
               ref_map(R['bkg'], R['xs'], R['ys'], x1 - x0, y1 - y0))


def test_run_parallel_end_to_end(cuda_dev, tmp_path):
    from caesar_yolo_b200 import weights as Wt
    from caesar_yolo_b200.inference import SFinder
    from caesar_yolo_b200.model import YOLO
    img = synth.make_mosaic(1024, 1536, seed=3, nan_border_frac=0.01)
    path = str(tmp_path / "m.fits")
    synth.write_fits(path, img, WCS_CARDS)
    model = YOLO(Wt.make_random_weights('n', 5, seed=0, cls_bias=-12.0))
    outs = []
    for k, maps in enumerate((False, True, True)):
        out = tmp_path / ("out%d" % k)
        out.mkdir()
        sf = SFinder(model, _config(path, str(out), True, save_bkg_maps=maps))
        assert sf.run_parallel() == 0
        outs.append(out)
    _same_outputs_plus_maps(outs[0], outs[1], 'm')
    nodes, bkg, rms, (X0, R0, W, H), rows = sf.engine.bkg_maps_band(sf.engine.tiles)
    assert (X0, R0, W, H) == (0, 0, 1536, 1024) and rows == (0, 1024)
    _check_files(str(outs[1]), 'm', W, H, X0, R0, bkg, rms)
    for a, b in zip(_map_files(str(outs[1]), 'm'), _map_files(str(outs[2]), 'm')):
        assert open(a, 'rb').read() == open(b, 'rb').read()
    R = ref_nodes(img, 101, 25)
    _check_nodes(nodes, R)
    _check_map(fits.FitsImage(_map_files(str(outs[1]), 'm')[1]).rows(0, H).astype(np.float32),
               ref_map(R['rms'], R['xs'], R['ys'], W, H))
