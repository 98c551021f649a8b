"""Drop-in for caesar_yolo/inference.py: `SFinder(model, config).run()` / `.run_parallel()` with the same config
dictionary, return codes (0 / -1) and output files, driven by the CUDA engine (pipeline.Engine).

Differences by design (B200-first): tiles are processed in batches on the GPU instead of one `model(...)` call per
tile; ranks are torch.distributed ranks (one per GPU) that own contiguous bands of tile rows instead of mpi4py
round-robin workers; the gather is one NCCL all-gather of 32-byte records; the neighbour table and both merges are
native/CUDA.  Catalog content and order equal the reference run with nproc=1."""
import json
import logging
import os
import time

import numpy as np
import torch

from . import catalog, fits as fitsmeta, inject, ops, reliability
from .fits import FitsImage
from .pipeline import Engine, make_pp_config, run_image
from .preprocessing import DataPreprocessor

logger = logging.getLogger(__name__)


def _dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def _as_sources(recs):
    """cy_det_record array -> cy_source array with the same boxes (what Engine.measure takes)."""
    src = np.zeros(len(recs), dtype=ops.SRC_DTYPE)
    for k in ('x1', 'y1', 'x2', 'y2', 'score', 'cls', 'flags', 'tile_id'):
        src[k] = recs[k]
    return src


def check_inject_options(n, rounds, snr_range):
    """Raises ValueError for an injection count < 0, rounds < 1 or an S/N range that is not (lo, hi), 0 < lo <= hi."""
    if n < 0:
        raise ValueError("inject_sources must be >= 0, not %d" % n)
    if rounds < 1:
        raise ValueError("inject_rounds must be >= 1, not %d" % rounds)
    if len(snr_range) != 2 or not (0 < snr_range[0] <= snr_range[1]) or not np.isfinite(snr_range[1]):
        raise ValueError("inject_snr_range must be (lo, hi) with 0 < lo <= hi, not %r" % (snr_range,))


class SFinder(object):
    """caesar_yolo/inference.py:280-1290."""

    def __init__(self, model, config):
        self.model = model
        self.config = config
        self.class_names = model.names
        self.sources = {"sources": []}
        self.results = {}
        self.outfile_json = config.get('outfile_json', '') if False else ''  # reference ignores the option (App. B#12)
        self.outfile_ds9 = ''
        self.write_to_json = config.get('save_catalog', True)
        self.write_to_ds9 = config.get('save_region', True)
        self.outdir = config.get('outdir', '.')
        self.save_tile_json = config.get('save_tile_catalog', False)
        self.save_tile_regions = config.get('save_tile_region', False)
        self.save_tile_img = config.get('save_tile_img', False)
        # per-source measurements (opt-in); the local noise needs the peak and sum of the box, so it implies them
        self.measure_noise = bool(config.get('measure_noise', False))
        self.measure_sources = bool(config.get('measure_sources', False)) or self.measure_noise
        self.noise_frame = int(config.get('noise_frame', 16))
        # the background-subtracted and S/N maps are made from the node states of the bkg / rms maps, so they imply them
        self.save_snr_maps = bool(config.get('save_snr_maps', False))
        self.save_bkg_maps = bool(config.get('save_bkg_maps', False)) or self.save_snr_maps
        self.bkg_box = int(config.get('bkg_box', 101))
        self.bkg_grid = int(config.get('bkg_grid', 25))
        # the catalog boxes masked out of the noise frames and the map nodes; only these two consumers use the mask
        self.bkg_mask_sources = bool(config.get('bkg_mask_sources', False))
        # completeness by injection and recovery: the injected S/N is set by the rms map of the same options
        self.inject_sources = int(config.get('inject_sources', 0))
        self.inject_rounds = int(config.get('inject_rounds', 1))
        self.inject_snr_range = tuple(float(v) for v in config.get('inject_snr_range', (3.0, 100.0)))
        self.inject_seed = int(config.get('inject_seed', 0))
        check_inject_options(self.inject_sources, self.inject_rounds, self.inject_snr_range)
        # reliability from the inverted image: the peak S/N of both catalogs is read from the S/N map of the same options
        self.reliability = bool(config.get('reliability', False))
        if self.bkg_mask_sources and not (self.measure_noise or self.save_bkg_maps or self.inject_sources or
                                          self.reliability):
            logger.warning("bkg_mask_sources masks the catalog boxes out of the measure_noise frames and the "
                           "save_bkg_maps nodes: with neither option on it changes nothing")
            self.bkg_mask_sources = False
        # the centre of the clipping of both consumers, so the per-source statistics and the maps still compare
        self.bkg_estimator = config.get('bkg_estimator', 'mean')
        if self.bkg_estimator not in ops.BKG_ESTIMATORS:
            raise ValueError("bkg_estimator must be one of %s, not %r" % (", ".join(ops.BKG_ESTIMATORS),
                                                                          self.bkg_estimator))
        if self.bkg_estimator != 'mean' and not (self.measure_noise or self.save_bkg_maps or self.inject_sources or
                                                 self.reliability):
            logger.warning("bkg_estimator sets the centre of the measure_noise and save_bkg_maps clipping: with neither "
                           "option on it changes nothing")
            self.bkg_estimator = 'mean'
        self.procId, self.nproc = _dist_info()
        self.timing = {}
        self.engine = None

    # ------------------------------------------------------------------------------------------------------
    def _pp_config(self):
        dp = self.config.get('preprocess_fcn')
        if dp is None:
            return make_pp_config(enabled=False)
        if isinstance(dp, DataPreprocessor):
            return dp.pp_config
        # any other callable (the reference's seam is "ndarray[H,W,3] -> ndarray[H,W,3] | None",
        # evaluation.py:157-161) runs on the host, tile by tile (_process_tiles_host_callable); the CUDA chain is off
        return make_pp_config(enabled=False)

    def _host_callable(self):
        dp = self.config.get('preprocess_fcn')
        return dp if (dp is not None and not isinstance(dp, DataPreprocessor)) else None

    def _process_tiles_host_callable(self, eng, tiles, ids, fcn):
        """Tiles through a foreign preprocess_fcn: TileTask.find_sources -> Analyzer.predict (inference.py:190-215,
        evaluation.py:128-193) with the callable on the HOST (it is the user's Python), everything after it on the GPU:
        letterbox + forward + decode / NMS + per-tile merge + records, one tile per launch sequence."""
        for tid in ids:
            t = tiles[int(tid)]
            x0, x1, y0, y1 = int(t['xmin']), int(t['xmax']), int(t['ymin']), int(t['ymax'])
            rows = self.fits.rows(y0, y1)
            data = np.array(rows[:, x0:x1], copy=True)
            if self.fits.is_raw_f32:
                data = data.view('>f4').astype(np.float32)
            data = data.astype(np.float64)
            data[~np.isfinite(data)] = 0                              # utils.py:219,394
            H, W = data.shape
            cube = np.zeros((H, W, 3))
            cube[:, :, 0] = cube[:, :, 1] = cube[:, :, 2] = data      # evaluation.py:146-154
            status = torch.zeros(1, dtype=torch.int32, device=eng.device)
            out = fcn(cube)
            if out is None or getattr(out, 'ndim', 0) != 3 or out.shape[2] != 3:
                status[0] = -1                                        # evaluation.py:164-166
                out = np.zeros((H, W, 3), np.float32)
            else:   # evaluation.py:171-176 (bug-compatible: image[i] is ROW i)
                if any(np.min(out[i]) == np.max(out[i]) for i in range(min(3, out.shape[0]))):
                    status[0] = -1
            H, W = out.shape[:2]
            x, _ = ops.letterbox_resize(torch.from_numpy(np.ascontiguousarray(out, dtype=np.float32)).to(eng.device)
                                        .unsqueeze(0), eng.imgsz, dtype=eng.model.dtype)
            Sh, Sw, lb = ops.letterbox_shape(H, W, eng.imgsz)
            eng._run_batch(x, status, torch.tensor([int(tid)], dtype=torch.int32, device=eng.device), H, W, Sh, Sw, lb)

    def _device(self):
        devs = self.config.get('devices') or ['cuda:0']
        d = str(devs[self.procId % len(devs)] if self.config.get('use_multi_gpu') else devs[0])
        if d == 'cpu':
            raise ops.CaesarB200Error("--devices=cpu: the B200 build has no CPU path (use cuda:N)")
        if 'LOCAL_RANK' in os.environ and self.nproc > 1:
            return torch.device('cuda:%d' % int(os.environ['LOCAL_RANK']))
        return torch.device(d if ':' in d else 'cuda:%s' % d)

    def _engine(self):
        if self.engine is None:
            weights = self.model.weights if hasattr(self.model, 'weights') else self.model
            dev = self._device()
            torch.cuda.set_device(dev)
            if self.nproc > 1:       # one process per GPU: node-local pinned staging and reader threads
                from .pipeline import bind_host_to_device_numa
                bind_host_to_device_numa(dev.index if dev.index is not None else 0)
            dm = self.model.device_model() if hasattr(self.model, 'device_model') else weights
            self.engine = Engine(dm, self._pp_config(), imgsz=self.config['img_size'],
                                 score_thr=self.config['score_thr'], iou_thr=self.config['iou_thr'],
                                 thr_soft=self.config['merge_overlap_iou_thr_soft'],
                                 thr_hard=self.config['merge_overlap_iou_thr_hard'], device=dev,
                                 batch_tiles=self.config.get('batch_tiles', 296),
                                 precision=self.config.get('precision'))
        return self.engine

    def set_img_size_params(self):
        """inference.py:354-477 (pixel geometry; the beam / WCS cards of the header are read by the per-source
        measurements, fits.beam_area_pix / fits.pixel_to_world)."""
        c = self.config
        self.image_id = os.path.splitext(os.path.basename(os.path.abspath(c['image_path'])))[0]
        if os.path.splitext(c['image_path'])[1] in ('.png', '.jpg'):   # inference.py:396-404: size from PIL
            try:
                from PIL import Image
                with Image.open(c['image_path'], mode='r') as im:
                    self.nx, self.ny = im.size
            except Exception as e:
                logger.error("Failed to read image size (err=%s)", e)
                return -1
            self.fits = None
            self.xmin, self.xmax, self.ymin, self.ymax = 0, self.nx - 1, 0, self.ny - 1
            return 0
        try:
            self.fits = FitsImage(self.config['image_path'])
        except Exception as e:
            logger.error("Failed to read image header (err=%s)", e)
            return -1
        xmin, xmax, ymin, ymax = c['image_xmin'], c['image_xmax'], c['image_ymin'], c['image_ymax']
        if xmin >= 0 and xmax >= 0 and ymin >= 0 and ymax >= 0 and not (xmin == xmax == ymin == ymax == 0):
            self.xmin, self.xmax, self.ymin, self.ymax = xmin, xmax, ymin, ymax
            self.nx, self.ny = xmax - xmin + 1, ymax - ymin + 1
        else:
            self.nx, self.ny = self.fits.nx, self.fits.ny
            self.xmin, self.xmax, self.ymin, self.ymax = 0, self.nx - 1, 0, self.ny - 1
        return 0

    # ------------------------------------------------------------------------------------------------------
    def run(self):
        """Single image (inference.py:485-552): the whole (sub-)image is one tile; outputs come from the Analyzer
        (out_<id>.json / out_<id>.reg, evaluation.py:216-234)."""
        if self.set_img_size_params() < 0:
            return -1
        c = self.config
        ext = os.path.splitext(c['image_path'])[1]
        if ext in ('.png', '.jpg'):
            return self._run_raster()
        if ext != '.fits':
            logger.error("Unsupported image format (%s) given!", ext)
            return -1
        full = all(v in (0, -1) for v in (c['image_xmin'], c['image_xmax'], c['image_ymin'], c['image_ymax']))
        if full:
            x0, x1, y0, y1 = 0, self.fits.nx, 0, self.fits.ny
        else:  # read_fits_crop: max EXCLUSIVE (utils.py:382)
            x0, x1, y0, y1 = c['image_xmin'], c['image_xmax'], c['image_ymin'], c['image_ymax']
            if min(x0, x1, y0, y1) < 0 or x1 <= x0 or y1 <= y0:
                return -1
        cov = self._inject_beam()
        if cov is False:
            return -1
        rel = self._reliability_on()
        eng = self._engine()
        tiles = np.zeros(1, dtype=ops.TILE_DTYPE)
        tiles[0] = (x0, x1, y0, y1)
        t0 = time.time()
        eng.begin(tiles)
        dev_img = None
        if self._host_callable() is None or self.measure_sources or self.save_bkg_maps:
            img = self.fits.rows(y0, y1)
            dev_img = torch.from_numpy(np.array(img, copy=True).view(np.int32)).to(eng.device)   # memmap rows are read-only
        if self._host_callable() is not None:
            self._process_tiles_host_callable(eng, tiles, [0], self._host_callable())
        else:
            eng.process_tiles(dev_img, self.fits.nx, self.fits.is_raw_f32, 0, y0, [0])
        packed, n = eng.finish()
        recs = packed.cpu().numpy().view(ops.REC_DTYPE)
        status = 0
        # predict() adds no offsets in the serial path (image_xmin/ymin default 0, inference.py:530)
        recs = recs.copy()
        recs['x1'] -= x0; recs['x2'] -= x0; recs['y1'] -= y0; recs['y2'] -= y0
        meas = None
        # one mask of the catalog boxes over the crop, for the frames and the map nodes alike
        mask = eng.source_mask(_as_sources(recs), x1 - x0, 0, y1 - y0) if self.bkg_mask_sources else None
        if self.measure_sources:   # in the coordinates of the catalog: the (sub-)image read, columns from x0
            args = (_as_sources(recs), dev_img[:, x0:], self.fits.nx, self.fits.is_raw_f32, 0, x1 - x0, 0, y1 - y0)
            m = eng.measure(*args)
            noise = eng.measure_noise(*args, frame=self.noise_frame, mask=mask,
                                      estimator=self.bkg_estimator) if self.measure_noise else None
            meas = self._measurements(m, self.fits.header, x0, y0, noise)
        nodes = None
        # the map region: the crop read, columns from x0
        margs = (None if dev_img is None else dev_img[:, x0:], self.fits.nx, self.fits.is_raw_f32, 0, x1 - x0, 0,
                 y1 - y0, 0, y1 - y0, self.bkg_box, self.bkg_grid)
        if self.save_bkg_maps:
            nodes, bkg, rms = eng.bkg_maps(*margs, mask=mask, estimator=self.bkg_estimator)
            region = (x0, y0, x1 - x0, y1 - y0)
            self._write_maps('bkg_maps_write_s', (('bkgmap_', bkg, True), ('rmsmap_', rms, True)), 0, region)
            del bkg, rms   # freed before res / snr are allocated: no more than two region maps at a time
            if self.save_snr_maps:
                res, snr = eng.snr_maps(nodes, *margs)
                self._write_maps('snr_maps_write_s', (('resmap_', res, True), ('snrmap_', snr, False)), 0, region)
        self.timing['run_s'] = time.time() - t0
        status = self._save_serial(recs, status, meas)
        crop = np.zeros(1, dtype=ops.TILE_DTYPE)
        crop[0] = (0, x1 - x0, 0, y1 - y0)

        def rerun(ids):
            if len(ids):
                eng.process_tiles(dev_img, self.fits.nx, self.fits.is_raw_f32, 0, y0, [0])

        def merge():
            p, _ = eng.finish()
            r = p.cpu().numpy().view(ops.REC_DTYPE).copy()
            r['x1'] -= x0; r['x2'] -= x0; r['y1'] -= y0; r['y2'] -= y0
            return _as_sources(r)
        if cov is not None:   # after every other output: the rounds change none of them
            t1 = time.time()
            if nodes is None:
                nodes, _, _ = eng.bkg_maps(*margs, mask=mask, estimator=self.bkg_estimator, maps=False)
            plan = inject.Plan(region=(0, 0, x1 - x0, y1 - y0), catalog=_as_sources(recs), tiles=crop, my_tiles=(0, 1),
                               target=margs[:7], x_off=0, centre_masked=self._centre_masked(x0, y0),
                               sample_rms=lambda cx, cy: eng.sample_bkg_maps(nodes, x1 - x0, 0, y1 - y0, self.bkg_box,
                                                                             self.bkg_grid, cx, cy)[1],
                               rerun=rerun, merge=merge)
            self._inject_rounds(plan, cov)
            self.timing['inject_s'] = time.time() - t1
        if rel:   # after every other output, the injection included: it changes none of them
            t1 = time.time()
            if nodes is None:
                nodes, _, _ = eng.bkg_maps(*margs, mask=mask, estimator=self.bkg_estimator, maps=False)
            plan = inject.Plan(catalog=_as_sources(recs), tiles=crop, my_tiles=(0, 1), target=margs[:7], rerun=rerun,
                               merge=merge, peak_snr=lambda src, sign: eng.peak_snr(nodes, src, *margs, sign=sign))
            self._reliability(plan, merged_key=False)
            self.timing['reliability_s'] = time.time() - t1
        return status

    # ------------------------------------------------------------------------------------------------------
    def _inject_beam(self):
        """C_pix of the beam when the run injects sources (fits.beam_cov_pix), None when it does not, False (after
        logging an error) when the header has no beam or pixel scale.  PNG / JPG input and a foreign preprocess_fcn
        (it reads its tiles from the file, so it would not see the injection) log one warning and inject nothing."""
        if not self.inject_sources:
            return None
        if self.fits is None:
            logger.warning("Source injection needs a FITS image: no injection into %s", self.config['image_path'])
            return None
        if self._host_callable() is not None:
            logger.warning("Source injection needs the CUDA preprocessing chain (a foreign preprocess_fcn reads its "
                           "tiles from the file and would not see the injected sources): no injection")
            return None
        cov = fitsmeta.beam_cov_pix(self.fits.header)
        if cov is None:
            logger.error("Source injection needs the beam (BMAJ, BMIN) and the pixel scale (CDELT or CD) in the image "
                         "header")
            return False
        return cov

    def _centre_masked(self, x0, y0):
        """centre_masked(cx, cy) of the injection placement: pixel (cx + x0, cy + y0) of the file is 0 or
        non-finite (decoded as the rows the run read)."""
        def f(cx, cy):
            v = np.asarray(self.fits.raw[np.asarray(cy) + y0, np.asarray(cx) + x0]).astype(np.float32)
            if not self.fits.is_raw_f32:
                v = v * np.float32(self.fits.bscale) + np.float32(self.fits.bzero)
            return ~np.isfinite(v) | (v == 0)
        return f

    def _inject_rounds(self, plan, cov):
        """inject.run_rounds on the plan; rank 0 writes inject_<image_id>.json.  The per-tile debug outputs are off
        during the rounds."""
        eng = self.engine
        keep = eng.tile_status, eng.tile_img_sink
        eng.tile_status, eng.tile_img_sink = None, None
        try:
            out = inject.run_rounds(eng, plan, self.inject_sources, self.inject_rounds, self.inject_snr_range,
                                    self.inject_seed, cov, self.class_names, rank=self.procId)
        finally:
            eng.tile_status, eng.tile_img_sink = keep
        if self.procId != 0:
            return
        params = {'seed': self.inject_seed, 'rounds': self.inject_rounds, 'n': self.inject_sources,
                  'snr_range': list(self.inject_snr_range), 'cov_pix': [[float(v) for v in row] for row in cov],
                  'footprint': list(inject.footprint_half(cov)), 'bkg_estimator': self.bkg_estimator,
                  'bkg_mask_sources': self.bkg_mask_sources, 'bkg_box': self.bkg_box, 'bkg_grid': self.bkg_grid}
        doc = inject.report(self.image_id, out[0], out[1], params)
        with open(os.path.join(self.outdir, 'inject_' + str(self.image_id) + '.json'), 'w') as f:
            json.dump(doc, f, indent=1)

    def _reliability_on(self):
        """True when the run estimates the reliability.  PNG / JPG input and a foreign preprocess_fcn (it reads its
        tiles from the file, so it would not see the negated rows) log one warning and estimate nothing."""
        if not self.reliability:
            return False
        if self.fits is None:
            logger.warning("The reliability estimate needs a FITS image: none for %s", self.config['image_path'])
            return False
        if self._host_callable() is not None:
            logger.warning("The reliability estimate needs the CUDA preprocessing chain (a foreign preprocess_fcn reads "
                           "its tiles from the file and would not see the inverted image): none")
            return False
        return True

    def _reliability(self, plan, merged_key):
        """reliability.run on the plan; rank 0 writes reliability_<image_id>.json and, with save_region,
        reliability_<image_id>.reg (the negative detections).  The per-tile debug outputs are off during the rerun."""
        eng = self.engine
        keep = eng.tile_status, eng.tile_img_sink
        eng.tile_status, eng.tile_img_sink = None, None
        try:
            neg, pos_peak, neg_peak = reliability.run(eng, plan)
        finally:
            eng.tile_status, eng.tile_img_sink = keep
        if self.procId != 0:
            return
        params = {'snr_range': list(self.inject_snr_range), 'score_thr': float(self.config['score_thr']),
                  'bkg_estimator': self.bkg_estimator, 'bkg_mask_sources': self.bkg_mask_sources,
                  'bkg_box': self.bkg_box, 'bkg_grid': self.bkg_grid}
        doc = reliability.report(self.image_id, plan.catalog, neg, pos_peak, neg_peak, self.class_names, params,
                                 len(plan.tiles))
        with open(os.path.join(self.outdir, 'reliability_' + str(self.image_id) + '.json'), 'w') as f:
            json.dump(doc, f, indent=1)
        if self.write_to_ds9:
            catalog.write_ds9(doc['negative_detections'],
                              os.path.join(self.outdir, 'reliability_' + str(self.image_id) + '.reg'),
                              merged_key=merged_key)

    def _measurements(self, m, header, x0=0, y0=0, noise=None):
        """Engine.measure output -> catalog.measurement_dicts with flux (beam area of the header) and the sky position
        of the centroid (SIN / TAN WCS; x0, y0: offset of the catalog's pixel grid in the file); noise: the
        Engine.measure_noise output of the same sources, or None."""
        radec = fitsmeta.pixel_to_world(header, m['xc'] + x0, m['yc'] + y0)
        if radec is None:
            logger.warning("No RA---SIN/TAN, DEC--SIN/TAN celestial WCS in the image header (CTYPE1=%s, CTYPE2=%s): "
                           "ra/dec are written as null", header.get('CTYPE1'), header.get('CTYPE2'))
        return catalog.measurement_dicts(m, fitsmeta.beam_area_pix(header), radec, noise)

    def _write_maps(self, timing_key, maps, row_begin, region):
        """<prefix><id>.fits in outdir for each (prefix, rows, bunit) of maps: this rank's map rows of the region
        (X0, R0, W, H), with the image's WCS shifted to the region; bunit=False leaves BUNIT out (a dimensionless
        map)."""
        X0, R0, W, H = region
        t0 = time.time()
        for name, rows, bunit in maps:
            hdr = fitsmeta.map_header(self.fits.header, W, H, X0, R0, bkgmask=self.bkg_mask_sources,
                                      bkgest=self.bkg_estimator, bunit=bunit)
            fitsmeta.write_map_rows(os.path.join(self.outdir, name + str(self.image_id) + '.fits'), hdr, rows,
                                    row_begin, W, H, self.procId, self.nproc)
        self.timing[timing_key] = time.time() - t0

    def _save_serial(self, recs, status, meas=None):
        self.results = {"image_id": self.image_id, "objs": catalog.records_to_objs(recs, self.class_names, meas=meas)}
        if self.write_to_json:
            catalog.write_json(self.results, os.path.join(self.outdir, 'out_' + str(self.image_id) + '.json'))
        if self.write_to_ds9:
            catalog.write_ds9(self.results['objs'], os.path.join(self.outdir, 'out_' + str(self.image_id) + '.reg'),
                              merged_key=False)
        return status

    def _run_raster(self):
        """PNG / JPG input of the serial path (inference.py:511-520): `plt.imread` semantics (read_raster), alpha
        channel dropped.  A 2-D image, or one whose three channels are equal, takes the same batched tile path as a
        FITS image (Analyzer.predict replicates a 2-D image into 3 channels, evaluation.py:146-154).  A colour image
        goes straight to the letterbox + model stages; the CUDA preprocessing chain works on one plane, so colour
        input together with --preprocessing is refused (-1) instead of being approximated."""
        from .fits import read_raster
        c = self.config
        try:
            a = read_raster(c['image_path'])
        except Exception as e:
            logger.error("Failed to read image %s (err=%s)", c['image_path'], e)
            return -1
        if a.ndim == 3 and a.shape[2] == 4:
            a = a[:, :, :3]
        if a.ndim == 3 and a.shape[2] != 3:
            logger.error("Unsupported channel count %d in %s", a.shape[2], c['image_path'])
            return -1
        gray = a.ndim == 2 or (np.array_equal(a[:, :, 0], a[:, :, 1]) and np.array_equal(a[:, :, 0], a[:, :, 2]))
        eng = self._engine()
        H, W = a.shape[:2]
        tiles = np.zeros(1, dtype=ops.TILE_DTYPE)
        tiles[0] = (0, W, 0, H)
        t0 = time.time()
        eng.begin(tiles)
        plane_dev = None
        if gray:
            plane = np.ascontiguousarray(a if a.ndim == 2 else a[:, :, 0], dtype=np.float32)
            plane[~np.isfinite(plane)] = 0
            plane_dev = torch.from_numpy(plane).to(eng.device)
            eng.process_tiles(plane_dev, W, False, 0, 0, [0])
        else:
            if eng.pp_cfg.nstages > 0:
                logger.error("Colour image with --preprocessing: the preprocessing chain of this build takes "
                             "single-plane images (FITS, grey PNG/JPG)")
                return -1
            cube = np.ascontiguousarray(a, dtype=np.float32)
            status = torch.zeros(1, dtype=torch.int32, device=eng.device)
            # evaluation.py:171-176 (bug-compatible: image[i] is ROW i): a constant row 0..2 rejects the image
            if any(cube[i].min() == cube[i].max() for i in range(min(3, H))):
                status[0] = -1
            x, _ = ops.letterbox_resize(torch.from_numpy(cube).to(eng.device).unsqueeze(0), eng.imgsz,
                                        dtype=eng.model.dtype)
            Sh, Sw, lb = ops.letterbox_shape(H, W, eng.imgsz)
            eng._run_batch(x, status, torch.zeros(1, dtype=torch.int32, device=eng.device), H, W, Sh, Sw, lb)
        packed, n = eng.finish()
        recs = packed.cpu().numpy().view(ops.REC_DTYPE).copy()
        meas = None
        if self.inject_sources:
            logger.warning("Source injection needs a FITS image: no injection into %s", c['image_path'])
        self._reliability_on()
        if self.save_bkg_maps:
            logger.warning("%s maps are written for FITS images only: none for %s",
                           "Background, rms, background-subtracted and S/N" if self.save_snr_maps
                           else "Background and rms", c['image_path'])
        if self.measure_sources:
            if plane_dev is None:
                logger.warning("Colour image: per-source measurements need a single-plane image and are not written")
            else:
                args = (_as_sources(recs), plane_dev, W, False, 0, W, 0, H)
                mask = eng.source_mask(args[0], W, 0, H) if self.bkg_mask_sources and self.measure_noise else None
                noise = eng.measure_noise(*args, frame=self.noise_frame, mask=mask,
                                          estimator=self.bkg_estimator) if self.measure_noise else None
                meas = self._measurements(eng.measure(*args), {}, noise=noise)
        self.timing['run_s'] = time.time() - t0
        return self._save_serial(recs, 0, meas)

    def run_parallel(self):
        """Tiled path (inference.py:578-658)."""
        t0 = time.time()
        if self.set_img_size_params() < 0:
            return -1
        if self.fits is None:   # tiles are cut with read_fits_crop in the reference (inference.py:190-195): FITS only
            logger.error("Tiled runs need a FITS image")
            return -1
        c = self.config
        tiles = ops.generate_tiles(self.xmin, self.xmax, self.ymin, self.ymax, c['tile_xsize'], c['tile_ysize'],
                                   c['tile_xstep'], c['tile_ystep'])
        if tiles is None:
            logger.error("Failed to generate tile grid")
            return -1
        T = len(tiles)
        ntasks_max = -(-T // self.nproc)
        if ntasks_max > c['max_ntasks_per_worker']:  # inference.py:1150-1160
            logger.error("Too many tasks per worker (%d > %d), increase --max_ntasks_per_worker or the GPU count",
                         ntasks_max, c['max_ntasks_per_worker'])
            return -1
        cov = self._inject_beam()
        if cov is False:
            return -1
        rel = self._reliability_on()
        eng = self._engine()
        img = self.fits   # raw big-endian float32 rows are read from the file into pinned staging (pipeline._RowSource)
        # per-tile debug files (inference.py:218-229): every rank writes the files of its own tiles
        hook = None
        eng.collect_tile_status = bool(self.save_tile_json or self.save_tile_regions)
        eng.tile_img_sink = None
        if self.save_tile_img:
            from .fits import write_fits

            def sink(tid, ch0):  # evaluation.py:550-554: image[:,:,0] (float64 in the reference)
                write_fits(ch0.astype(np.float64),
                           os.path.join(self.outdir, 'timg_' + str(self.image_id) + '_tid' + str(tid) + '.fits'))
            eng.tile_img_sink = sink
        if eng.collect_tile_status:
            def hook(packed, n, a, b):
                recs = packed[:n * 32].cpu().numpy().view(ops.REC_DTYPE)
                st = eng.tile_status[a:b].cpu().numpy()
                catalog.write_tile_outputs(recs, tiles, np.arange(a, b), st, self.class_names, self.image_id,
                                           self.outdir, self.save_tile_json, self.save_tile_regions)
        # measurements, masked maps, injection and reliability need the catalog on every rank (each measures or masks
        # its own rows)
        rank0_only = not (self.measure_sources or (self.save_bkg_maps and self.bkg_mask_sources) or cov is not None or
                          rel)
        if self._host_callable() is not None:
            from .pipeline import split_tile_rows
            eng.begin(tiles)
            a, b = split_tile_rows(tiles, self.nproc)[self.procId]
            eng._my_range = (a, b)
            self._process_tiles_host_callable(eng, tiles, range(a, b), self._host_callable())
            src, n = eng.exchange_and_merge(self.nproc, rank0_only=rank0_only, rank=self.procId,
                                            on_local_records=hook)
            # the tiles went through the host: bring this rank's rows to the GPU
            if self.measure_sources or self.save_bkg_maps:
                Y0, Y1 = (int(tiles['ymin'][a:b].min()), int(tiles['ymax'][a:b].max())) if b > a else (0, 0)
                band = torch.from_numpy(np.array(self.fits.rows(Y0, Y1), copy=True).view(np.int32)).to(eng.device)
                eng.band = (band if b > a else None, Y0, Y1, self.fits.nx, self.fits.is_raw_f32)
        else:
            src, n = run_image(eng, img, self.fits.is_raw_f32, tiles, rank=self.procId, world=self.nproc,
                               on_rank0_only=rank0_only, on_local_records=hook)
        meas = None
        nodes = None
        # one mask of the catalog boxes over this rank's rows, for the frames and the map nodes alike
        mask = eng.source_mask_band(src, tiles, self.procId, self.nproc) if self.bkg_mask_sources else None
        if self.measure_sources:
            m = eng.measure_band(src, tiles, self.procId, self.nproc)
            noise = None
            if self.measure_noise:
                noise = eng.measure_noise_band(src, tiles, self.noise_frame, self.procId, self.nproc, mask=mask,
                                               estimator=self.bkg_estimator)
            if self.procId == 0:
                meas = self._measurements(m, self.fits.header, noise=noise)
        if self.save_bkg_maps:   # every rank maps and writes its own rows; unmasked maps need no catalog
            nodes, bkg, rms, region, rows = eng.bkg_maps_band(tiles, self.bkg_box, self.bkg_grid, self.procId,
                                                              self.nproc, mask=mask, estimator=self.bkg_estimator)
            self._write_maps('bkg_maps_write_s', (('bkgmap_', bkg, True), ('rmsmap_', rms, True)),
                             rows[0] - region[1], region)
            del bkg, rms   # freed before res / snr are allocated: no more than two region maps at a time
            if self.save_snr_maps:   # the same rows of the band, no collective
                res, snr, _, _ = eng.snr_maps_band(nodes, tiles, self.bkg_box, self.bkg_grid, self.procId, self.nproc)
                self._write_maps('snr_maps_write_s', (('resmap_', res, True), ('snrmap_', snr, False)),
                                 rows[0] - region[1], region)
        self.timing['run_s'] = time.time() - t0
        if self.procId == 0:
            self.sources = {"sources": catalog.sources_to_dicts(src, self.class_names, meas)}
            self.save()
            logger.info("Run completed in %d seconds", int(time.time() - t0))
        if cov is not None:   # after every other output: the rounds change none of them
            t1 = time.time()
            if nodes is None:
                nodes = eng.bkg_maps_band(tiles, self.bkg_box, self.bkg_grid, self.procId, self.nproc, mask=mask,
                                          estimator=self.bkg_estimator, maps=False)[0]
            plan = inject.tiled_plan(eng, tiles, src, nodes, self.bkg_box, self.bkg_grid, self._centre_masked(0, 0),
                                     self.procId, self.nproc)
            self._inject_rounds(plan, cov)
            self.timing['inject_s'] = time.time() - t1
        if rel:   # after every other output, the injection included: it changes none of them
            t1 = time.time()
            if nodes is None:
                nodes = eng.bkg_maps_band(tiles, self.bkg_box, self.bkg_grid, self.procId, self.nproc, mask=mask,
                                          estimator=self.bkg_estimator, maps=False)[0]
            plan = reliability.tiled_plan(eng, tiles, src, nodes, self.bkg_box, self.bkg_grid, self.procId, self.nproc)
            self._reliability(plan, merged_key=True)
            self.timing['reliability_s'] = time.time() - t1
        return 0

    def save(self):
        """inference.py:1167-1194."""
        if self.procId != 0:
            return
        if self.write_to_json:
            catalog.write_json(self.sources, os.path.join(self.outdir, 'catalog_' + str(self.image_id) + '.json'))
        if self.write_to_ds9:
            catalog.write_ds9(self.sources['sources'], os.path.join(self.outdir, 'ds9_' + str(self.image_id) + '.reg'))
