"""Host-side driver of the B200 hot path: FITS mosaic -> tiles -> preprocessing -> YOLOv8 forward -> decode/NMS ->
per-tile merge -> records -> (all-gather) -> cross-tile merge -> catalog.  Python only orchestrates; every stage is a
CUDA kernel behind the C ABI (ops.py)."""
from ._capi import PPChain, PPConfig


def make_pp_config(enabled=True, subtract_bkg=False, sigma_bkg=3.0, use_box_mask_in_bkg=False, bkg_box_mask_fract=0.7,
                   bkg_chid=-1, clip_shift_data=False, sigma_clip=1.0, clip_chid=-1, clip_data=False,
                   sigma_clip_low=10.0, sigma_clip_up=10.0, nchannels=1, zscale_stretch=False,
                   zscale_contrasts=(0.25, 0.25, 0.25), chan3_preproc=False, sigma_clip_baseline=0.0,
                   normalize_minmax=False, norm_min=0.0, norm_max=1.0, out_f16=False):
    """cy_pp_config from the run.py option names and defaults (scripts/run.py:80-107, stage order :272-293)."""
    c = PPConfig()
    c.enabled = 1 if enabled else 0
    c.subtract_bkg = int(bool(subtract_bkg))
    c.sigma_bkg = float(sigma_bkg)
    c.use_box_mask_in_bkg = int(bool(use_box_mask_in_bkg))
    c.bkg_box_mask_fract = float(bkg_box_mask_fract)
    c.bkg_chid = int(bkg_chid)
    c.clip_shift_data = int(bool(clip_shift_data))
    c.sigma_clip = float(sigma_clip)
    c.clip_chid = int(clip_chid)
    c.clip_data = int(bool(clip_data))
    c.sigma_clip_low = float(sigma_clip_low)
    c.sigma_clip_up = float(sigma_clip_up)
    c.nchannels = int(nchannels)
    c.zscale_stretch = int(bool(zscale_stretch))
    zc = list(zscale_contrasts) + [0.25] * 3
    for i in range(3):
        c.zscale_contrasts[i] = float(zc[i])
    c.chan3_preproc = int(bool(chan3_preproc))
    c.sigma_clip_baseline = float(sigma_clip_baseline)
    c.normalize_minmax = int(bool(normalize_minmax))
    c.norm_min = float(norm_min)
    c.norm_max = float(norm_max)
    c.out_f16 = 1 if out_f16 else 0
    return c


# ======================================================================================================= engine

import os
import time

from typing import NamedTuple

import numpy as np
import torch

from . import ops
from ._capi import CaesarB200Error, Letterbox


class SourceMask(NamedTuple):
    """Engine.source_mask: the bit mask of rows [row_begin, row_end) (int32 device tensor [rows, ceil(ncols / 32)],
    layout: ops.source_mask) and the columns and rows it was built over, which its consumers check."""
    bits: torch.Tensor
    ncols: int
    row_begin: int
    row_end: int


class Engine(object):
    """One GPU's share of the hot path.  Holds the device model and reusable buffers; `process_tiles` runs
    preprocessing -> forward -> decode/NMS -> per-tile merge -> records for a list of tiles cut out of an image that
    is already in device memory; `finish` compacts the records; `global_merge` builds the catalog.

    Replaces TileTask.find_sources + Analyzer.predict (caesar_yolo/inference.py:173-275, evaluation.py:128-245) for
    all tiles of a rank at once (the reference runs them one by one, batch 1)."""

    def __init__(self, weights, pp_cfg, imgsz=640, score_thr=0.7, iou_thr=0.5, thr_soft=0.3, thr_hard=0.8,
                 device=None, batch_tiles=296, pp_tiles=296, precision=None):
        if not torch.cuda.is_available():
            raise CaesarB200Error("no CUDA device: the B200 path has no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        torch.cuda.set_device(self.device)
        ops.check(ops.lib.cy_device_check())
        self.model = weights if isinstance(weights, ops.DeviceModel) else ops.DeviceModel(weights, precision=precision)
        self.nc = self.model.nc
        self.names = self.model.names
        src_cfg = pp_cfg if pp_cfg is not None else make_pp_config(enabled=False)
        # private copy of the stage list (a cy_pp_config is expanded to run.py's stage order): the output format
        # follows the model
        if isinstance(src_cfg, PPChain):
            self.pp_cfg = ops.validate_chain(PPChain.from_buffer_copy(src_cfg))
        else:
            self.pp_cfg = ops.chain_from_config(src_cfg)
        self.pp_cfg.out_f16 = 1 if self.model.dtype == torch.float16 else 0
        self.imgsz = int(imgsz)
        self.score_thr, self.iou_thr = float(score_thr), float(iou_thr)
        self.thr_soft, self.thr_hard = float(thr_soft), float(thr_hard)
        self.batch_tiles = int(batch_tiles)
        self.pp_tiles = max(int(pp_tiles), self.batch_tiles)
        self._buf = {}
        self.launches = 0      # kernels launched by this engine (bench.py's gpu_launches)
        self.stage_events = None   # set to [] to collect (stage, start_event, end_event) triples (bench breakdown)
        self._fwd_launches = {}
        # per-tile debug outputs (--save_tile_catalog / --save_tile_region / --save_tile_img, inference.py:218-229):
        self.collect_tile_status = False   # keep the per-tile status (0 ok, <0 rejected) in self.tile_status
        self.tile_img_sink = None          # callable(tile_id, ndarray[Ty,Tx] float32): channel 0 after the chain

    def _mark(self):
        if self.stage_events is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _stage(self, name, e0):
        if e0 is not None:
            self.stage_events.append((name, e0, self._mark()))

    def stage_times_ms(self):
        """Sum of CUDA-event durations per stage since stage_events was last reset (synchronises)."""
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.stage_events or []:
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out

    # ---- buffers -----------------------------------------------------------------------------------------
    def _get(self, key, shape, dtype):
        t = self._buf.get(key)
        n = int(np.prod(shape))
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty((n,), dtype=dtype, device=self.device)
            self._buf[key] = t
        return t[:n].view(*shape)

    def begin(self, tiles):
        """tiles: structured array (ops.TILE_DTYPE) of ALL tiles of the mosaic (global ids = row-major index)."""
        self.tiles = np.ascontiguousarray(tiles)
        self.T = len(tiles)
        self.tiles_dev = ops.to_device_bytes(self.tiles, self.device)
        self.rec_slots = self._get('rec_slots', (self.T * ops.MAX_DET * 32,), torch.uint8)
        self.nrec = self._get('nrec', (self.T,), torch.int32)
        self.nrec.zero_()
        self.launches += 1
        self._my_range = (0, self.T)
        self.tile_status = None
        self.band = None          # (device rows, first row, end row, columns, big_endian) of the last run_image
        if self.collect_tile_status:
            self.tile_status = torch.full((self.T,), -3, dtype=torch.int32, device=self.device)  # -3: not processed

    def process_tiles(self, img_dev, row_stride, big_endian, origin_x, origin_y, tile_ids, ready=None, min_groups=1):
        """img_dev covers mosaic rows/cols starting at (origin_x, origin_y); tile_ids: global ids of the tiles to
        process (all must lie inside img_dev).  Groups by tile shape (edge tiles are smaller, SURVEY App. B#24).
        Preprocessing runs in groups of `pp_tiles` tiles (one CTA per tile: a multiple of the SM count keeps all 148
        SMs busy); the conv stack and the detect/merge kernels run in batches of `batch_tiles`.
        ready(y): optional callback invoked before a group is launched, y = last mosaic row (exclusive) the group
        reads (run_image uses it to wait for / issue the upload of those rows)."""
        tile_ids = np.asarray(tile_ids, dtype=np.int32)
        if tile_ids.size == 0:
            return
        t = self.tiles[tile_ids]
        w = t['xmax'] - t['xmin']
        h = t['ymax'] - t['ymin']
        shapes = sorted(set(zip(h.tolist(), w.tolist())), reverse=True)
        for (Ty, Tx) in shapes:
            ids = tile_ids[(h == Ty) & (w == Tx)]
            starts = list(range(0, len(ids), self.pp_tiles))
            if min_groups > 1:
                # host-staged input: a small LEADING group (whole tile rows, >= 32 tiles) starts computing as soon as
                # its rows are in HBM; the upload of everything else overlaps it
                lead = lead_group_size(self.tiles['ymin'][ids], LEAD_TILES)
                if 0 < lead and 2 * lead <= len(ids):
                    starts = [0] + list(range(lead, len(ids), self.pp_tiles))
            for k, s in enumerate(starts):
                g = ids[s:(starts[k + 1] if k + 1 < len(starts) else len(ids))]
                if ready is not None:
                    ready(int(self.tiles['ymax'][g].max()))
                self._run_group(img_dev, row_stride, big_endian, origin_x, origin_y, g, Ty, Tx)

    def _run_group(self, img_dev, row_stride, big_endian, ox, oy, ids, Ty, Tx):
        G = len(ids)
        dev = self.device
        tl = self.tiles[ids]
        meta = np.concatenate([(tl['xmin'] - ox).astype(np.int32), (tl['ymin'] - oy).astype(np.int32),
                               ids.astype(np.int32)])
        meta_dev = torch.from_numpy(meta).to(dev, non_blocking=True)
        x0, y0, ids_dev = meta_dev[:G], meta_dev[G:2 * G], meta_dev[2 * G:]
        Sh, Sw, lb = ops.letterbox_shape(Ty, Tx, self.imgsz)
        want_chain = self.tile_img_sink is not None
        chain = self._get('chain', (G, Ty, Tx, 3), torch.float32) if want_chain else None
        model_in = self._get('model_in', (G, Sh, Sw, 4), self.model.dtype)
        status = self._get('pp_status', (G,), torch.int32)
        need = int(ops.lib.cy_preprocess_chain_scratch_bytes(ops.ctypes.byref(self.pp_cfg), G, Ty, Tx))
        scratch = self._get('pp_scratch', (need,), torch.uint8)
        e = self._mark()
        ops.preprocess(self.pp_cfg, img_dev, row_stride, big_endian, x0, y0, Ty, Tx, self.imgsz, scratch=scratch,
                       chain_out=chain, model_in=model_in, status=status, want_chain=want_chain)
        self._stage('preprocess', e)
        self.launches += 4        # bucket, chain, geometry, fused final
        if self.tile_img_sink is not None:   # Analyzer.write_fits: channel 0 of the preprocessed image, accepted tiles
            ok = status.cpu().numpy()
            ch0 = chain[:, :, :, 0].cpu().numpy()
            for k in range(G):
                if ok[k] == 0:
                    self.tile_img_sink(int(ids[k]), ch0[k])
        for s in range(0, G, self.batch_tiles):
            e = min(G, s + self.batch_tiles)
            self._run_batch(model_in[s:e], status[s:e], ids_dev[s:e], Ty, Tx, Sh, Sw, lb)

    def _run_batch(self, model_in, status, ids_dev, Ty, Tx, Sh, Sw, lb):
        B = model_in.shape[0]
        dev = self.device
        key = (B, Ty, Tx)
        lbd = self._buf.get(('lb',) + key)
        if lbd is None:
            lbd = ops.letterbox_array([lb] * B, dev)
            self._buf[('lb',) + key] = lbd
        e = self._mark()
        heads = self.model.forward(model_in)
        self._stage('forward', e)
        e = self._mark()
        need = int(ops.lib.cy_postprocess_scratch_bytes(B, Sh, Sw, ops.MAX_DET))
        pscr = self._get('post_scratch', (need,), torch.uint8)
        dets = self._get('dets', (B, ops.MAX_DET, 6), torch.float32)
        ndets = self._get('ndets', (B,), torch.int32)
        ops.postprocess(heads, B, Sh, Sw, self.nc, self.score_thr, self.iou_thr, lbd, dev, scratch=pscr, dets=dets,
                        ndets=ndets)
        self._stage('decode_nms', e)
        e = self._mark()
        keep = self._get('keep', (B, ops.MAX_DET), torch.int32)
        nkeep = self._get('nkeep', (B,), torch.int32)
        mstat = self._get('mstat', (B,), torch.int32)
        ops.merge_tile(dets, ndets, self.score_thr, self.thr_soft, self.thr_hard, keep_idx=keep, nkeep=nkeep,
                       status=mstat, pre_status=status)
        ops.make_records(dets, keep, nkeep, mstat, self.tiles_dev, ids_dev, self.rec_slots, self.nrec)
        self._stage('merge_tile_records', e)
        if self.tile_status is not None:
            self.tile_status.index_copy_(0, ids_dev.long(), mstat)
        fl = self._fwd_launches.get((B, Sh, Sw))
        if fl is None:
            fl = int(self.model.info(B, Sh, Sw)['launches'])
            self._fwd_launches[(B, Sh, Sw)] = fl
        # forward + memset/score/nms (3) + merge + records (2)
        self.launches += fl + 3 + 2

    def pp_kernels(self):
        """Names of the preprocessing kernels cy_preprocess launches for this configuration (bench.py's roofline)."""
        return ("pp_bucket_kernel + pp_chain_kernel + pp_geom_kernel + pp_fused4_kernel (pp_fused_kernel for tiles whose "
                "interleaved planes do not fit shared memory)")

    def finish(self):
        """Compacts the per-tile record slots -> (packed uint8 tensor of n cy_det_record, n) in tile-id order.
        Synchronises (n is read on the host); the exchange path below does not use it."""
        packed = self._compact_local()
        n = int(self._buf['total'][0].item())
        return packed[:n * 32], n

    def _compact_local(self):
        """Device-only: record slots -> self._buf['packed'] in tile-id order, count in self._buf['total'] (int32[1])."""
        total = self._get('total', (8,), torch.int32)          # [0] = count; padded to one 32-byte record
        packed = self._get('packed', (self.T * ops.MAX_DET * 32,), torch.uint8)
        scr = self._get('compact_scratch', (int(ops.lib.cy_compact_scratch_bytes(self.T)),), torch.uint8)
        ops.compact_records(self.rec_slots, self.nrec, self.T, ops.MAX_DET, packed, total, scratch=scr)
        self.launches += 4
        return packed

    def neighbor_csr(self):
        """Device CSR of the tile neighbour lists of the CURRENT tile grid (rebuilt when begin() saw another grid)."""
        key = self.tiles.tobytes()
        cached = self._buf.get('nb')
        if cached is None or cached[0] != key:
            nb_off, nb_idx = ops.tile_neighbors(self.tiles)
            cached = (key, torch.from_numpy(nb_off).to(self.device),
                      torch.from_numpy(nb_idx if len(nb_idx) else np.zeros(1, np.int32)).to(self.device))
            self._buf['nb'] = cached
        return cached[1], cached[2]

    def global_merge(self, packed, n, nb_off=None, nb_idx=None):
        """find_sources_at_edge + merge_edge_sources -> numpy structured array (ops.SRC_DTYPE)."""
        if nb_off is None:
            off_dev, idx_dev = self.neighbor_csr()
        else:
            off_dev = torch.from_numpy(nb_off).to(self.device)
            idx_dev = torch.from_numpy(nb_idx if len(nb_idx) else np.zeros(1, np.int32)).to(self.device)
        out = self._get('sources', (max(n, 1) * 32,), torch.uint8)
        self.launches += 33
        e = self._mark()
        res = ops.merge_global(packed, n, self.tiles_dev, self.T, off_dev, idx_dev, out=out)
        self._stage('merge_global', e)
        return res

    def exchange_and_merge(self, world, rank0_only=False, rank=0, on_local_records=None):
        """Exchange step + catalog assembly (SFinder.gather_task_data_from_workers + find_sources_at_edge +
        merge_edge_sources, inference.py:936-984,663-931).  Every rank compacts its records on the device into a
        fixed-capacity slot [count | cap records], ONE all-gather moves all slots, a second device compaction builds the
        tile-id-ordered list; the host reads a single scalar (the total) before the merge.  Returns (sources, n)."""
        e = self._mark()
        packed = self._compact_local()
        if on_local_records is not None:
            n_loc = int(self._buf['total'][0].item())
            on_local_records(packed, n_loc, *self._my_range)
        if world == 1:
            n = int(self._buf['total'][0].item())
            self._stage('exchange', e)
            return self.global_merge(packed[:n * 32], n), n
        import torch.distributed as dist
        cap = self._exchange_cap(world)
        while True:
            send = self.pack_send(packed, cap)
            recv = self._get('xrecv', (world * (cap + 1) * 32,), torch.uint8)
            dist.all_gather_into_tensor(recv, send)
            allp, n, cmax = self.unpack_recv(recv, world, cap)
            if cmax <= cap:
                break
            cap = self._exchange_cap(world, need=cmax)                  # a rank overflowed its slot: grow and redo
        self._stage('exchange', e)
        if rank0_only and rank != 0:
            return None, n
        return self.global_merge(allp[:n * 32], n), n

    def pack_send(self, packed, cap):
        """This rank's all-gather slot: one 32-byte header (record count in its first int32) + the first `cap` records."""
        send = self._get('xsend', ((cap + 1) * 32,), torch.uint8)
        send[:32].copy_(self._buf['total'][:8].view(torch.uint8))
        send[32:].copy_(packed[:cap * 32])
        self.launches += 2
        return send

    def unpack_recv(self, recv, world, cap):
        """Gathered slots [world, cap + 1 records] -> (records of all ranks in rank = tile-id order, total, largest
        per-rank count).  Device compaction; the return values cost the one host read of the exchange."""
        counts = recv.view(torch.int32).view(world, (cap + 1) * 8)[:, 0].contiguous()
        allp = self._get('xall', (world * cap * 32,), torch.uint8)
        tot = self._get('xtotal', (8,), torch.int32)
        scr = self._get('xscratch', (int(ops.lib.cy_compact_scratch_bytes(world)),), torch.uint8)
        ops.compact_records(recv[32:], counts.clamp(max=cap), world, cap + 1, allp, tot, scratch=scr)
        self.launches += 8
        h = torch.cat([tot[:1], counts.max().view(1)]).cpu()
        return allp, int(h[0]), int(h[1])

    def measure(self, sources, img, row_stride, big_endian, row0, ncols, row_begin, row_end, world=1):
        """Per-source measurements of the catalog `sources` (ops.SRC_DTYPE) over rows [row_begin, row_end) of `img`, a
        device tensor of 4-byte pixels whose first element is image row row0, column 0 (cy_measure_sources).  With
        world > 1 every rank passes the same catalog and its own rows: the partials are all-gathered in the group of the
        record exchange and folded in rank order (cy_measure_combine).  Returns a structured array (ops.MEAS_DTYPE)."""
        src = np.ascontiguousarray(sources, dtype=ops.SRC_DTYPE)
        n = len(src)
        if n == 0:
            return np.zeros(0, dtype=ops.MEAS_DTYPE)
        src_dev = ops.to_device_bytes(src, self.device)
        e = self._mark()
        part = ops.measure_sources(img, row_stride, big_endian, row0, ncols, src_dev, n, row_begin, row_end,
                                   out=self._get('meas_part', (n * ops.PARTIAL_BYTES,), torch.uint8))
        if world > 1:
            import torch.distributed as dist
            allp = self._get('meas_gather', (world * n * ops.PARTIAL_BYTES,), torch.uint8)
            dist.all_gather_into_tensor(allp, part)
        else:
            allp = part
        meas = ops.measure_combine(allp, world, src_dev, n, ncols)
        self._stage('measure', e)
        self.launches += 4 + (1 if world > 1 else 0)
        return meas.cpu().numpy().view(ops.MEAS_DTYPE)

    def measure_band(self, sources, tiles, rank=0, world=1):
        """Engine.measure over the rows this rank owns (measure_rows), read from the band of mosaic rows the last
        run_image left in HBM: no second read of the file."""
        r0, r1 = measure_rows(tiles, world)[rank]
        band, Y0, _, nx, big_endian = self.band
        if band is None:                     # a rank without tiles still takes part in the all-gather
            band, Y0 = self._get('meas_noband', (1,), torch.int32), r0
        return self.measure(sources, band, nx, big_endian, Y0, nx, r0, r1, world=world)

    def source_mask(self, sources, ncols, row_begin, row_end):
        """Bit mask of the union of the boxes of the catalog `sources` (ops.SRC_DTYPE) over columns [0, ncols) and rows
        [row_begin, row_end) (cy_source_mask; layout: ops.source_mask) -> SourceMask.  A run builds it once over the rows
        it measures and passes it to measure_noise and bkg_maps, so both leave the catalog boxes out of their
        statistics."""
        src = np.ascontiguousarray(sources, dtype=ops.SRC_DTYPE)
        e = self._mark()
        out = torch.empty((row_end - row_begin, ops.source_mask_words(ncols)), dtype=torch.int32, device=self.device)
        mask = ops.source_mask(ops.to_device_bytes(src, self.device), len(src), ncols, row_begin, row_end, out=out)
        self._stage('source_mask', e)
        self.launches += 3 if len(src) else 1
        return SourceMask(mask, ncols, row_begin, row_end)

    def source_mask_band(self, sources, tiles, rank=0, world=1):
        """Engine.source_mask over the image columns and the rows this rank owns (measure_rows): the mask that
        measure_noise_band and bkg_maps_band take."""
        r0, r1 = measure_rows(tiles, world)[rank]
        return self.source_mask(sources, self.band[3], r0, r1)

    def measure_noise(self, sources, img, row_stride, big_endian, row0, ncols, row_begin, row_end, frame=16, world=1,
                      mask=None, estimator='mean'):
        """Local background and noise of the catalog `sources` (ops.SRC_DTYPE): sigma-clipped mean / std of a frame of
        `frame` pixels around each box, over rows [row_begin, row_end) of `img` (arguments as for Engine.measure;
        cy_noise_init / cy_noise_pass / cy_noise_update).  One pass per clipping iteration, at most
        ops.NOISE_MAX_PASSES; with world > 1 every rank passes the same catalog and its own rows, and the partials of
        each pass are all-gathered in the group of the record exchange.  Every rank folds the same partials, so every
        rank sees the same active count and runs the same passes.  mask: Engine.source_mask of the same catalog, ncols
        and rows, or None; with it, the frame pixels inside any catalog box are masked (cy_noise_pass_masked).  Returns
        a structured array (ops.NOISE_DTYPE) whose bkg, rms, nbkg, iters are final; self.noise_passes holds the number
        of passes run.  estimator: 'mean' (mean-centred clipping) or 'median' (median-centred, bkg = the median of the
        last set; every pass is ops.SELECT_ROUNDS rounds, see Engine._median_passes)."""
        _check_estimator('Engine.measure_noise', estimator)
        src = np.ascontiguousarray(sources, dtype=ops.SRC_DTYPE)
        n = len(src)
        self.noise_passes = 0
        if n == 0:
            return np.zeros(0, dtype=ops.NOISE_DTYPE)
        if mask is not None and (mask.ncols, mask.row_begin, mask.row_end) != (ncols, row_begin, row_end):
            raise CaesarB200Error("Engine.measure_noise: a mask of %d columns, rows [%d, %d) for a frame of %d columns, "
                                  "rows [%d, %d)" % (mask.ncols, mask.row_begin, mask.row_end, ncols, row_begin,
                                                     row_end))
        src_dev = ops.to_device_bytes(src, self.device)
        e = self._mark()
        state = self._get('noise_state', (n * ops.NOISE_DTYPE.itemsize,), torch.uint8)
        off = self._get('noise_off', (n + 1,), torch.int64)
        units = ops.noise_init(src_dev, n, ncols, row_begin, row_end, frame, state, off)
        part = self._get('noise_part', (n * ops.NOISE_PARTIAL_BYTES,), torch.uint8)
        allp = part
        if world > 1:
            import torch.distributed as dist
            allp = self._get('noise_gather', (world * n * ops.NOISE_PARTIAL_BYTES,), torch.uint8)
        if estimator == 'median':
            def run_round(sel, rnd, hist):
                ops.noise_pass_median(img, row_stride, big_endian, row0, ncols, src_dev, n, row_begin, row_end, frame,
                                      off, units, state, sel, rnd, part, hist, None if mask is None else mask.bits)
            self.noise_passes = self._median_passes('noise', n, state, part, allp, world, run_round, 'sources')
            self._stage('noise', e)
            self.launches += 3 + self.noise_passes * (9 + (5 if world > 1 else 0))
            return state.cpu().numpy().view(ops.NOISE_DTYPE)
        active = n
        while active:
            if self.noise_passes == ops.NOISE_MAX_PASSES:
                raise ops.CaesarB200Error("cy_noise_update: %d sources still active after %d passes"
                                          % (active, self.noise_passes))
            if mask is None:
                ops.noise_pass(img, row_stride, big_endian, row0, ncols, src_dev, n, row_begin, row_end, frame, off,
                               units, state, part)
            else:
                ops.noise_pass_masked(img, row_stride, big_endian, row0, ncols, src_dev, n, row_begin, row_end, frame,
                                      off, units, state, part, mask.bits)
            if world > 1:
                dist.all_gather_into_tensor(allp, part)
            active = ops.noise_update(allp, world, n, state)
            self.noise_passes += 1
        self._stage('noise', e)
        self.launches += 3 + self.noise_passes * (3 + (1 if world > 1 else 0))
        return state.cpu().numpy().view(ops.NOISE_DTYPE)

    def _median_passes(self, tag, n, state, part, allp, world, run_round, what):
        """Median-centred clipping passes of n sources or nodes until none is active: each pass is ops.SELECT_ROUNDS
        digit rounds of run_round(sel, rnd, hist) and cy_median_update.  With world > 1 the round-0 moment partials
        are all-gathered (folded in rank order, as for the mean) and the uint32 histograms are summed with one
        all-reduce per round: integer sums are exact in any order.  The active count is read once per pass.  Returns
        the number of passes."""
        sel = self._get(tag + '_sel', (n * ops.SELECT_BYTES,), torch.uint8)
        hist = self._get(tag + '_hist', (n * ops.SELECT_SLOTS,), torch.int32)
        if world > 1:
            import torch.distributed as dist
        passes, active = 0, n
        while active:
            if passes == ops.NOISE_MAX_PASSES:
                raise ops.CaesarB200Error("cy_median_update: %d %s still active after %d passes"
                                          % (active, what, passes))
            for rnd in range(ops.SELECT_ROUNDS):
                run_round(sel, rnd, hist)
                if world > 1:
                    if rnd == 0:
                        dist.all_gather_into_tensor(allp, part)
                    dist.all_reduce(hist)
                active = ops.median_update(allp, world, hist, n, state, sel, rnd)
            passes += 1
        return passes

    def measure_noise_band(self, sources, tiles, frame=16, rank=0, world=1, mask=None, estimator='mean'):
        """Engine.measure_noise over the rows this rank owns (measure_rows), read from the band of mosaic rows the last
        run_image left in HBM.  The frames are thus clipped to the rows the run read, and no rank reads a row twice.
        mask: Engine.source_mask_band of the same catalog, or None; estimator as for Engine.measure_noise."""
        r0, r1 = measure_rows(tiles, world)[rank]
        band, Y0, _, nx, big_endian = self.band
        if band is None:                     # a rank without tiles still takes part in every all-gather
            band, Y0 = self._get('meas_noband', (1,), torch.int32), r0
        return self.measure_noise(sources, band, nx, big_endian, Y0, nx, r0, r1, frame=frame, world=world, mask=mask,
                                  estimator=estimator)

    def bkg_maps(self, img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box=101, grid=25, world=1,
                 mask=None, mask_col0=0, estimator='mean'):
        """Background and rms maps of the region of columns [0, ncols) of `img` and rows [R0, R1) (node lattice,
        statistic and interpolation: include/caesar_b200.h), over rows [row_begin, row_end) of `img` (arguments as for
        Engine.measure; cy_bkg_grid_init / cy_bkg_grid_pass / cy_noise_update / cy_bkg_grid_maps).  With world > 1 every
        rank passes the same region and its own rows, and the node partials of each pass are all-gathered in the group of
        the record exchange, so every rank runs the same passes.  mask: Engine.source_mask of rows [row_begin, row_end),
        region column x being mask column x + mask_col0, or None.  With it, the node-box pixels inside any catalog box
        are masked (cy_bkg_grid_pass_masked), and the nodes left without a pixel whose box holds data are filled from
        their neighbours (cy_bkg_grid_probe_init, one unmasked pass of the probe, cy_bkg_grid_fill); self.bkg_holes_filled
        holds their count.  Returns (nodes, bkg, rms): the final node states (ops.NOISE_DTYPE, shape [Ny, Nx]) and this
        range's map rows as int32 device tensors [row_end - row_begin, ncols] holding big-endian float32;
        self.bkg_passes holds the number of clipping passes run.  estimator: as for Engine.measure_noise, so the maps and
        the per-source statistics of one run compare directly."""
        _check_estimator('Engine.bkg_maps', estimator)
        nx, ny = len(ops.bkg_grid_nodes(ncols, grid)), len(ops.bkg_grid_nodes(R1 - R0, grid))
        nodes = nx * ny
        if mask is not None and (mask.row_end - mask.row_begin != row_end - row_begin or
                                 (row_end > row_begin and mask.row_begin != row_begin)):
            raise CaesarB200Error("Engine.bkg_maps: a mask of rows [%d, %d) for rows [%d, %d)"
                                  % (mask.row_begin, mask.row_end, row_begin, row_end))
        e = self._mark()
        state = self._get('bkg_state', (nodes * ops.NOISE_DTYPE.itemsize,), torch.uint8)
        off = self._get('bkg_off', (ny + 1,), torch.int64)
        units = ops.bkg_grid_init(ncols, R0, R1, row_begin, row_end, box, grid, state, off)
        part = self._get('bkg_part', (nodes * ops.NOISE_PARTIAL_BYTES,), torch.uint8)
        allp = part
        if world > 1:
            import torch.distributed as dist
            allp = self._get('bkg_gather', (world * nodes * ops.NOISE_PARTIAL_BYTES,), torch.uint8)
        self.bkg_passes = 0
        active = 0 if estimator == 'median' else nodes
        if estimator == 'median':
            def run_round(sel, rnd, hist):
                ops.bkg_grid_pass_median(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid,
                                         off, units, state, sel, rnd, part, hist,
                                         None if mask is None else mask.bits, 0 if mask is None else mask.ncols,
                                         mask_col0)
            self.bkg_passes = self._median_passes('bkg', nodes, state, part, allp, world, run_round, 'grid nodes')
            self.launches += self.bkg_passes * (6 + (4 if world > 1 else 0))   # the rounds beyond the mean's pass
        while active:
            if self.bkg_passes == ops.NOISE_MAX_PASSES:
                raise ops.CaesarB200Error("cy_noise_update: %d grid nodes still active after %d passes"
                                          % (active, self.bkg_passes))
            if mask is None:
                ops.bkg_grid_pass(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid, off,
                                  units, state, part)
            else:
                ops.bkg_grid_pass_masked(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box,
                                         grid, off, units, state, part, mask.bits, mask.ncols, mask_col0)
            if world > 1:
                dist.all_gather_into_tensor(allp, part)
            active = ops.noise_update(allp, world, nodes, state)
            self.bkg_passes += 1
        self.bkg_holes_filled = 0
        if mask is not None:   # the node states are the same on every rank, and so is the probe count
            probe = self._get('bkg_probe', (nodes * ops.NOISE_DTYPE.itemsize,), torch.uint8)
            if ops.bkg_grid_probe_init(state, nodes, probe):
                ops.bkg_grid_pass(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid, off,
                                  units, probe, part)
                if world > 1:
                    dist.all_gather_into_tensor(allp, part)
                self.bkg_holes_filled = ops.bkg_grid_fill(allp, world, nx, ny, state)
                self.launches += 3 + (1 if world > 1 else 0) + 2
            self.launches += 1
        bkg = torch.empty((row_end - row_begin, ncols), dtype=torch.int32, device=self.device)
        rms = torch.empty_like(bkg)
        ops.bkg_grid_maps(state, ncols, R0, R1, row_begin, row_end, box, grid, bkg, rms)
        self._stage('bkg_maps', e)
        self.launches += 3 + self.bkg_passes * (3 + (1 if world > 1 else 0)) + 1
        return state.cpu().numpy().view(ops.NOISE_DTYPE).reshape(ny, nx), bkg, rms

    def bkg_maps_band(self, tiles, box=101, grid=25, rank=0, world=1, mask=None, estimator='mean'):
        """Engine.bkg_maps of the bounding box of the tile grid (columns [min xmin, max xmax), rows [min ymin,
        max ymax)) over the rows this rank owns (measure_rows), read from the band of mosaic rows the last run_image
        left in HBM.  mask: Engine.source_mask_band (image columns, so the region starts at its column X0), or None;
        estimator as for Engine.bkg_maps.
        Returns (nodes, bkg, rms, (X0, R0, W, H), (row_begin, row_end))."""
        img, nx, big_endian, Y0, (X0, R0, W, H), (r0, r1) = self._map_band(tiles, rank, world)
        nodes, bkg, rms = self.bkg_maps(img, nx, big_endian, Y0, W, R0, R0 + H, r0, r1, box, grid, world, mask=mask,
                                        mask_col0=X0, estimator=estimator)
        return nodes, bkg, rms, (X0, R0, W, H), (r0, r1)

    def _map_band(self, tiles, rank, world):
        """The map region of a tiled run, (X0, R0, W, H): the bounding box of the tile grid; this rank's rows of it
        (measure_rows, [R0, R0) when it has none); and where they are read: (img, row_stride, big_endian, row0, region,
        rows), img being the band of mosaic rows the last run_image left in HBM from column X0."""
        X0, X1 = int(tiles['xmin'].min()), int(tiles['xmax'].max())
        R0, R1 = int(tiles['ymin'].min()), int(tiles['ymax'].max())
        r0, r1 = measure_rows(tiles, world)[rank]
        if r1 == r0:
            r0 = r1 = R0
        band, Y0, _, nx, big_endian = self.band
        if band is None:                     # a rank without tiles still takes part in every all-gather
            img, Y0 = self._get('meas_noband', (1,), torch.int32), r0
        else:
            img = band[:, X0:]
        return img, nx, big_endian, Y0, (X0, R0, X1 - X0, R1 - R0), (r0, r1)

    def snr_maps(self, nodes, img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box=101, grid=25):
        """Background-subtracted and S/N maps (definition: include/caesar_b200.h) of the region of Engine.bkg_maps over
        rows [row_begin, row_end) of `img` (the same arguments), from `nodes`, the final node states Engine.bkg_maps
        returned (cy_bkg_grid_snr_maps).  One pass over the rows and no collective: each rank maps its own rows.
        Returns (res, snr): int32 device tensors [row_end - row_begin, ncols] holding big-endian float32."""
        nx, ny = len(ops.bkg_grid_nodes(ncols, grid)), len(ops.bkg_grid_nodes(R1 - R0, grid))
        nodes = np.ascontiguousarray(nodes, dtype=ops.NOISE_DTYPE)
        if nodes.shape != (ny, nx):
            raise CaesarB200Error("Engine.snr_maps: node states of shape %s for a lattice of %d x %d nodes"
                                  % (nodes.shape, ny, nx))
        e = self._mark()
        res = torch.empty((row_end - row_begin, ncols), dtype=torch.int32, device=self.device)
        snr = torch.empty_like(res)
        ops.bkg_grid_snr_maps(ops.to_device_bytes(nodes, self.device), img, row_stride, big_endian, row0, ncols, R0, R1,
                              row_begin, row_end, box, grid, res, snr)
        self._stage('snr_maps', e)
        self.launches += 1
        return res, snr

    def snr_maps_band(self, nodes, tiles, box=101, grid=25, rank=0, world=1):
        """Engine.snr_maps of the region and rows of Engine.bkg_maps_band (the same band of mosaic rows in HBM, so the
        file is not read again), from the node states it returned.  Returns (res, snr, (X0, R0, W, H), (row_begin,
        row_end))."""
        img, nx, big_endian, Y0, (X0, R0, W, H), (r0, r1) = self._map_band(tiles, rank, world)
        res, snr = self.snr_maps(nodes, img, nx, big_endian, Y0, W, R0, R0 + H, r0, r1, box, grid)
        return res, snr, (X0, R0, W, H), (r0, r1)

    def _exchange_cap(self, world, need=0):
        """Records per rank slot of the all-gather: 48 per tile of the largest band (the catalogs of the synthetic
        mosaics hold ~20 per tile), grown on demand; kept across steps so the buffers are allocated once."""
        cap = self._buf.get('xcap', 0)
        base = 48 * (-(-self.T // world)) + 1024
        want = max(cap, base, int(need * 1.25) + 1)
        want = min(want, self.T * ops.MAX_DET)
        self._buf['xcap'] = want
        return want


def _check_estimator(fn, estimator):
    if estimator not in ops.BKG_ESTIMATORS:
        raise CaesarB200Error("%s: estimator %r is not one of %s" % (fn, estimator, ", ".join(ops.BKG_ESTIMATORS)))


def piece_end(r0, y_end, rows_per_piece, y_stop):
    """Last row (exclusive) of the upload piece that starts at row r0: at most rows_per_piece rows, never past the band
    end y_end, and cut at y_stop — the last row the tile group waiting for this upload reads — when that falls inside
    the piece, so that the group waits for no byte it does not need."""
    r1 = min(y_end, r0 + rows_per_piece)
    if r0 < y_stop < r1:
        r1 = y_stop
    return r1


LEAD_TILES = int(os.environ.get('CY_LEAD_TILES', '32'))   # smallest leading group of a host-staged run (tuning knob)


def lead_group_size(ymins, min_tiles=32):
    """Tiles of the leading group of a host-staged run: the first whole tile rows that hold at least `min_tiles` tiles
    (ymins: ymin of the tiles in id order = row-major)."""
    n = len(ymins)
    k = 0
    while k < n:
        y = ymins[k]
        while k < n and ymins[k] == y:
            k += 1
        if k >= min_tiles:
            return k
    return 0


def measure_rows(tiles, world):
    """Row range [r0, r1) of the mosaic each rank measures, from the first row of its band (split_tile_rows) to the first
    row of the next rank's band; the last rank's range ends with its band.  The ranges partition the rows the run read,
    in rank order, and each lies inside its rank's band at any tile step, so a hull that crosses a band boundary is
    measured in parts with no halo.  A rank without tiles gets an empty range."""
    parts = split_tile_rows(tiles, world)
    bands = [(int(tiles['ymin'][a:b].min()), int(tiles['ymax'][a:b].max())) if b > a else None for a, b in parts]
    out = []
    for r, bd in enumerate(bands):
        if bd is None:
            out.append((0, 0))
            continue
        nxt = next((b2[0] for b2 in bands[r + 1:] if b2 is not None), bd[1])
        out.append((bd[0], max(bd[0], min(nxt, bd[1]))))
    return out


def bind_host_to_device_numa(device_index):
    """Pins the calling process to the CPUs of the NUMA node the GPU hangs off (sysfs), so that the pinned staging
    buffers it allocates afterwards are node-local (first touch) and the reader threads run next to them: with one
    process per GPU and every rank uploading its band at the same time, remote-node staging halves the H2D rate.
    Returns the node (or None when the topology is not visible: nothing is changed then)."""
    try:
        pr = torch.cuda.get_device_properties(device_index)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(','):
            if '-' in part:
                a, b = part.split('-')
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def split_tile_rows(tiles, nparts):
    """Partition of the row-major tile grid into `nparts` contiguous bands of whole tile rows, balanced by tile count.
    Returns list of (first_tile_id, last_tile_id_exclusive).  (Replaces the reference's round-robin tile->rank map,
    inference.py:1008-1029; the gathered list stays in tile-id order for any rank count.)"""
    T = len(tiles)
    ymins = tiles['ymin']
    row_starts = [0] + [i for i in range(1, T) if ymins[i] != ymins[i - 1]] + [T]
    nrows = len(row_starts) - 1
    parts = []
    for r in range(nparts):
        a = row_starts[(nrows * r) // nparts]
        b = row_starts[(nrows * (r + 1)) // nparts]
        parts.append((a, b))
    return parts


def allgather_records(packed, n, world_size):
    """Exchange step of the path on HOST-known counts (replaces SFinder.gather_task_data_from_workers,
    inference.py:936-984): all-gather of the fixed 32-byte detection records (counts first, then records padded to the
    max count — NCCL has no all-gather-v).  Ranks own ascending contiguous tile-id ranges, so concatenating in rank
    order keeps the list in tile-id order, i.e. the reference's nproc=1 order, for any world size.  Works on CUDA
    tensors over NCCL and on CPU tensors over gloo (tests); the GPU pipeline uses Engine.exchange_and_merge, which
    keeps the counts on the device."""
    import torch.distributed as dist
    if world_size == 1:
        return packed, n
    dev = packed.device
    cnt = torch.tensor([n], dtype=torch.int32, device=dev)
    counts = [torch.zeros(1, dtype=torch.int32, device=dev) for _ in range(world_size)]
    dist.all_gather(counts, cnt)
    counts = [int(c.item()) for c in counts]
    mx = max(max(counts), 1)
    send = torch.zeros((mx * 32,), dtype=torch.uint8, device=dev)
    send[:n * 32] = packed[:n * 32]
    if dev.type == 'cuda':
        recv = torch.empty((world_size * mx * 32,), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(recv, send)
        parts = [recv[r * mx * 32: r * mx * 32 + counts[r] * 32] for r in range(world_size)]
    else:
        bufs = [torch.empty((mx * 32,), dtype=torch.uint8) for _ in range(world_size)]
        dist.all_gather(bufs, send)
        parts = [bufs[r][:counts[r] * 32] for r in range(world_size)]
    return torch.cat(parts), sum(counts)


# ---------------------------------------------------------------------------------------------- host row sources

READ_THREADS = 8
_read_pool = None


def _pool():
    global _read_pool
    if _read_pool is None:
        from concurrent.futures import ThreadPoolExecutor
        _read_pool = ThreadPoolExecutor(max_workers=READ_THREADS)
    return _read_pool


class _RowSource(object):
    """Rows [r0, r1) of the mosaic as a pinned int32 tensor view ready for an asynchronous H2D copy."""

    def __init__(self, engine, img_host, nx, rows_per_piece):
        self.eng, self.img, self.nx, self.rpp = engine, img_host, nx, rows_per_piece
        self.is_torch = isinstance(img_host, torch.Tensor)
        self.fd = None
        self.offset = 0
        if not self.is_torch and hasattr(img_host, 'path') and getattr(img_host, 'is_raw_f32', False):
            self.fd = os.open(img_host.path, os.O_RDONLY)          # FitsImage: read the payload rows straight from the file
            self.offset = int(img_host.offset)
        elif not self.is_torch and hasattr(img_host, 'rows'):
            self.img = img_host.rows(0, img_host.ny)                # scaled / integer FITS payloads: converted on the host

    def close(self):
        if self.fd is not None:
            os.close(self.fd)
            self.fd = None

    def _staging(self, k, nwords):
        slot = ('pin', k & 1)
        pin, ev = self.eng._buf.get(slot, (None, None))
        if pin is None or pin.numel() < nwords:
            pin = torch.empty((max(self.rpp * self.nx, nwords),), dtype=torch.int32, pin_memory=True)
            ev = None
        if ev is not None:
            ev.synchronize()                                        # the previous DMA out of this buffer has completed
        return slot, pin

    def get(self, k, r0, r1):
        """-> (pinned tensor [r1-r0, nx] int32, staging slot or None)."""
        if self.is_torch:
            src = self.img[r0:r1]
            return (src.view(torch.int32) if src.dtype != torch.int32 else src), None
        nwords = (r1 - r0) * self.nx
        slot, pin = self._staging(k, nwords)
        dst = pin[:nwords].numpy().view(np.uint8)
        if self.fd is not None:
            read_file_range(self.fd, self.offset + r0 * self.nx * 4, dst)
        else:
            np.copyto(dst.reshape(r1 - r0, self.nx * 4),
                      np.ascontiguousarray(self.img[r0:r1]).view(np.uint8).reshape(r1 - r0, self.nx * 4))
        self.eng._buf[slot] = (pin, None)
        return pin[:nwords].view(r1 - r0, self.nx), slot


def read_file_range(fd, offset, dst_u8):
    """preadv of len(dst_u8) bytes at `offset` into a writable uint8 numpy view, split over READ_THREADS threads (the
    system call releases the GIL, so the page-cache / disk reads run in parallel)."""
    n = dst_u8.size
    nt = READ_THREADS if n >= (8 << 20) else 1
    step = -(-n // nt)
    step = (step + 4095) & ~4095

    def one(i):
        a, b = i * step, min(n, (i + 1) * step)
        mv = memoryview(dst_u8[a:b])
        done = 0
        while done < b - a:
            got = os.preadv(fd, [mv[done:]], offset + a + done)
            if got <= 0:
                raise IOError("short read from the FITS payload")
            done += got
    parts = [i for i in range(nt) if i * step < n]
    if len(parts) == 1:
        one(0)
    else:
        list(_pool().map(one, parts))


def read_rows_benchmark(engine, fimg, y0, y1, piece_bytes=1 << 26):
    """Reads rows [y0, y1) of a FitsImage payload into the engine's pinned staging buffers with the reader run_image
    uses, nothing else running (bench.py reports the rate next to the file-inclusive throughput).  Returns bytes read."""
    nx = fimg.nx
    rpp = max(1, int(piece_bytes) // (nx * 4))
    src = _RowSource(engine, fimg, nx, rpp)
    torch.cuda.synchronize()
    total, k, r = 0, 0, y0
    try:
        while r < y1:
            r1 = min(y1, r + rpp)
            src.get(k, r, r1)
            total += (r1 - r) * nx * 4
            r, k = r1, k + 1
    finally:
        src.close()
    return total


def run_image(engine, img_host, big_endian, tiles, rank=0, world=1, piece_bytes=1 << 26, on_rank0_only=True,
              on_local_records=None):
    """FITS payload on the HOST -> catalog.  img_host: a pinned torch tensor [ny,nx] of 4-byte pixels (zero-copy
    staging), a numpy array / memmap, or a fits.FitsImage (rows are read from the file with preadv into pinned staging
    buffers); big_endian: raw FITS byte order.  The rows of this rank's tiles (contiguous band of tile rows) are
    uploaded in pieces of ~piece_bytes on a copy stream; every tile group waits only for the rows it needs, so all but
    the first group's read + upload overlap the compute of earlier groups; the first group is kept small (the first
    whole tile rows with >= 32 tiles) so that little of the upload is exposed.
    on_local_records(packed, n, first_tile_id, last_tile_id_excl): called with this rank's records before the exchange
    (per-tile output files).  Returns (sources structured array or None on ranks != 0, n_records_total)."""
    engine.begin(tiles)
    a, b = split_tile_rows(tiles, world)[rank]
    engine._my_range = (a, b)
    ids = np.arange(a, b, dtype=np.int32)
    if isinstance(img_host, torch.Tensor):
        ny, nx = img_host.shape[0], img_host.shape[1]
    elif hasattr(img_host, 'nx') and hasattr(img_host, 'ny'):
        ny, nx = img_host.ny, img_host.nx
    else:
        ny, nx = img_host.shape[0], img_host.shape[1]
    if len(ids):
        Y0, Y1 = int(tiles['ymin'][ids].min()), int(tiles['ymax'][ids].max())
        copy_stream = engine._buf.get('copy_stream')
        if copy_stream is None:
            copy_stream = torch.cuda.Stream(device=engine.device)
            engine._buf['copy_stream'] = copy_stream
        compute = torch.cuda.current_stream()
        band = engine._get('band', (Y1 - Y0, nx), torch.int32)   # reused across calls: no allocation per image
        copy_stream.wait_stream(compute)                          # earlier work may still read the band buffer
        rows_per_piece = max(1, int(piece_bytes) // (nx * 4))
        src = _RowSource(engine, img_host, nx, rows_per_piece)
        state = {'row': Y0, 'events': []}                         # events[i] = (last_row_excl, event)

        def upload_piece(y_stop):
            r0 = state['row']
            r1 = piece_end(r0, Y1, rows_per_piece, y_stop)
            k = len(state['events'])
            rows, slot = src.get(k, r0, r1)
            with torch.cuda.stream(copy_stream):
                band[r0 - Y0:r1 - Y0].copy_(rows, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            if slot is not None:
                engine._buf[slot] = (engine._buf[slot][0], ev)
            state['events'].append((r1, ev))
            state['row'] = r1

        def ready(y_needed):
            """Called before a tile group is launched: rows [Y0, y_needed) must be in HBM."""
            while state['row'] < min(y_needed, Y1):
                upload_piece(min(y_needed, Y1))
            for r1, ev in state['events']:
                if r1 >= min(y_needed, Y1):
                    compute.wait_event(ev)
                    break

        try:
            engine.process_tiles(band, nx, big_endian, 0, Y0, ids, ready=ready, min_groups=2)
        finally:
            src.close()
        engine.band = (band, Y0, Y1, nx, bool(big_endian))
    else:
        engine.band = (None, 0, 0, nx, bool(big_endian))
    return engine.exchange_and_merge(world, rank0_only=on_rank0_only, rank=rank, on_local_records=on_local_records)
