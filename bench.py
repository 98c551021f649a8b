#!/usr/bin/env python
"""bench.py — headline benchmark of the caesar-yolo hot path on B200 (contract: see the task prompt).

Workloads (SURVEY.md §8d numbering, `--config`):
  3 (default, BASELINE.json configs[2]): synthetic 16384 x 16384 float32 radio mosaic (FITS payload byte order),
    512 x 512 tiles at step 1.0 -> 1024 tiles, random-init YOLOv8l (nc=5, seeded), imgsz 640, full preprocessing chain
    (subtract_bkg, clip_data, zscale_stretch, chan3_preproc, normalize_minmax), FITS payload -> merged catalog.
  4 (configs[3]): the same generator at 32768 x 32768 (seed 5678), step 0.5 -> 16 384 tiles (cross-tile merge stress).
  5 (configs[4]): 256 synthetic imgsz-1024 head-map tiles, scoreThr 0.05, ~10 k candidates per tile through Detect
    decode -> NMS -> per-tile merge only (dense-candidate NMS stress).
One "step" = one full pass mosaic -> catalog.  N GPUs split the SAME mosaic into contiguous bands of tile rows
(strong scaling), exchange 32-byte detection records with one NCCL all-gather and merge on every rank.

  value    : tiles/s with the mosaic band already resident in HBM (device timed, max over ranks)
  e2e      : the same through the host-facing call with the mosaic in pinned HOST memory: H2D of the payload and D2H of
             the catalog inside the timed region
  e2e_file : the same starting from the FITS FILE on local disk (read + staging + H2D inside the timed region)
  --impl reference : the CPU oracle (restatement of the reference's --devices=cpu path) on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault('NCCL_DEBUG', 'INFO')   # communicator evidence for the driver; fd 1 is kept clean below

# The contract is ONE JSON line on stdout.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
# log there), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a private duplicate of the
# original stdout.
_JSON_OUT = None


def claim_stdout():
    """Called once by main(): keeps a private handle on the real stdout and sends everything else to stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


PP_FLAGS = dict(subtract_bkg=True, clip_data=True, zscale_stretch=True, chan3_preproc=True, normalize_minmax=True,
                nchannels=3, norm_max=255.)
SCORE_THR, IOU_THR, SOFT, HARD = 0.5, 0.5, 0.3, 0.8
CLS_BIAS = {'n': -16.0, 'l': -24.0, '11n': -20.0, '11l': -24.0}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', type=int, default=3, choices=[3, 4, 5],
                    help='SURVEY §8d workload: 3 = 16k mosaic step 1.0 (BASELINE configs[2], headline), 4 = 32k mosaic '
                         'step 0.5 (configs[3]), 5 = dense-candidate NMS stress (configs[4])')
    ap.add_argument('--mosaic', type=int, default=None)
    ap.add_argument('--tile', type=int, default=512)
    ap.add_argument('--step', type=float, default=None)
    ap.add_argument('--variant', default='l')
    ap.add_argument('--imgsz', type=int, default=640)
    ap.add_argument('--batch', type=int, default=296)
    ap.add_argument('--precision', default=None, choices=['fp16', 'bf16'],
                    help='16-bit storage of weights / activations (default: the package default, fp16)')
    ap.add_argument('--cpu-tiles', type=int, default=16, help='tiles in the bounded CPU-baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-profile', action='store_true')
    ap.add_argument('--no-file', action='store_true', help='skip the FITS-file-inclusive measurement')
    ap.add_argument('--no-alt', action='store_true', help='skip the informational run in the other 16-bit format')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the timed path returned in its last timed step as DIR/<name>.npy (float32 / '
                         'float64; integer fields as float64) so that two builds can be compared output for output: '
                         'the merged catalog (the same for any GPU count), or with --config 5 the outputs of rank 0\'s '
                         '256 tiles (the same head maps for any GPU count; other ranks draw their own)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.mosaic is None:
        a.mosaic = 32768 if a.config == 4 else 16384
    if a.step is None:
        a.step = 0.5 if a.config == 4 else 1.0
    return a


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for k, nme in enumerate(names):
                    if r[4 + k].lower().startswith('active'):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('hbm_gbs', 6650.0), d.get('bf16_tflops_sustained', 1400.0), d.get('bf16_tflops', 1590.0), 'measured'
    return 6650.0, 1400.0, 1590.0, 'fallback'


def mosaic_seed(n):
    return 1234 if n <= 16384 else 5678


def make_mosaic_pinned(args):
    """Synthetic mosaic in raw FITS payload order (big-endian float32) in pinned host memory."""
    import torch
    from caesar_yolo_b200 import synth
    n = args.mosaic
    img = synth.make_mosaic(n, n, seed=mosaic_seed(n), nan_border_frac=0.0)
    b = int(0.02 * n)
    img[-b:, :] = np.nan           # 2% NaN strips (bottom/right: NaN top rows make the reference reject those tiles)
    img[:, -b:] = np.nan
    host = torch.empty((n, n), dtype=torch.int32, pin_memory=True)
    hv = host.numpy().view(np.uint32)
    rows = max(1, (1 << 24) // n)
    for y0 in range(0, n, rows):
        hv[y0:y0 + rows] = img[y0:y0 + rows].view(np.uint32).byteswap()
    return img, host


def count_tiles(size, tile, step):
    """len(utils.generate_tiles) for a square image (caesar_yolo/utils.py:622-697), without loading any library."""
    st = int(round(step * tile))
    n1 = len(range(0, size, st))
    return n1 * n1


def sample_side(args):
    return args.tile * int(np.ceil(np.sqrt(args.cpu_tiles)))


def cpu_reference(args, sub, threads, keep_catalog=False):
    """The oracle (restated reference --devices=cpu path) on the sub-mosaic `sub`, as a FITS file -> catalog run of
    oracle.SFinder.run_parallel.  Returns (tiles/s, seconds, tiles, catalog list or None)."""
    import tempfile
    import torch
    from caesar_yolo_b200 import synth, weights as W
    from oracle import inference as oinf, preprocessing as opp, yolo as oy
    torch.set_num_threads(threads)
    tmp = tempfile.mkdtemp(prefix='cybench_')
    path = os.path.join(tmp, 'sub.fits')
    synth.write_fits(path, sub)
    w = W.make_random_weights(args.variant, 5, seed=0, cls_bias=CLS_BIAS.get(args.variant, -16.0))
    dp = opp.DataPreprocessor(opp.build_stages(**PP_FLAGS))
    cfg = dict(img_size=args.imgsz, preprocess_fcn=dp, image_path=path, image_xmin=-1, image_xmax=-1, image_ymin=-1,
               image_ymax=-1, mpi=None, split_image_in_tiles=True, tile_xsize=args.tile, tile_ysize=args.tile,
               tile_xstep=args.step, tile_ystep=args.step, max_ntasks_per_worker=1 << 30, devices=['cpu'],
               iou_thr=IOU_THR, merge_overlap_iou_thr_soft=SOFT, merge_overlap_iou_thr_hard=HARD, score_thr=SCORE_THR,
               save_catalog=True, outdir=tmp)
    model = oy.OracleModel(w)
    sf = oinf.SFinder(model, cfg)
    t0 = time.time()
    sf.run_parallel()
    dt = time.time() - t0
    nt = len(sf.tasks_per_worker[0])
    return nt / dt, dt, nt, (sf.sources['sources'] if keep_catalog else None)


def run_reference(args):
    """Reference arm: the oracle port of the reference's CPU path on a bounded sample.  Never touches the product
    library (no caesar_yolo_b200.ops / _capi import: synth and weights are pure numpy / torch)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    from caesar_yolo_b200 import synth
    threads = os.cpu_count() or 1
    n = sample_side(args)
    img = synth.make_mosaic(n, n, seed=1234, nan_border_frac=0.0)
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, nt, cat = cpu_reference(args, img, threads, keep_catalog=bool(args.dump_outputs))
        if i >= args.warmup:
            vals.append((v, dt, nt))
    if args.dump_outputs:      # the oracle's catalog under the field names of the b200 dump (it has no tile ids)
        out = {'sources_' + k: np.array([s[k] for s in cat], np.float64) for k in ('x1', 'y1', 'x2', 'y2', 'score')}
        out['sources_cls'] = np.array([s['class_id'] for s in cat])
        out['sources_flags'] = np.array([int(bool(s['edge'])) | 2 * int(bool(s.get('merged', False))) for s in cat])
        dump_outputs(args.dump_outputs, out)
    v = float(np.mean([x[0] for x in vals]))
    ms = float(np.mean([x[1] for x in vals])) * 1e3
    nt = vals[0][2]
    sample = ("%d tiles (%dx%d mosaic of the same generator), oracle SFinder.run_parallel FITS->catalog, torch CPU fp32 "
              "batch 1 per tile, logging silenced" % (nt, n, n))
    cfg = workload_config(args, args.gpus, T=nt, mosaic=n)
    cfg["sampled_from"] = ("bounded sample of the %dx%d workload (%d tiles): the reference's O(T^2) Python neighbour "
                           "search and per-tile batch-1 CPU forward make the full mosaic impractical"
                           % (args.mosaic, args.mosaic, count_tiles(args.mosaic, args.tile, args.step)))
    line = {"impl": "reference", "metric": "tiles/s FITS->catalog", "value": v, "unit": "tiles/s", "n_gpus": args.gpus,
            "steps": len(vals), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "tiles/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mpix_per_s": v * args.tile * args.tile / 1e6}
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs, "outputs": "oracle catalog of the %d-tile sample" % nt}
    emit(line)
    return 0


def workload_config(args, n, T=None, mosaic=None):
    mosaic = args.mosaic if mosaic is None else mosaic
    if T is None:
        T = count_tiles(mosaic, args.tile, args.step)
    return {"workload": "synthetic %dx%d f32 mosaic (FITS byte order), %dx%d tiles step %.1f (%d tiles), %s nc=5 "
                        "random-init, imgsz %d, full preprocessing chain, FITS payload -> merged catalog"
                        % (mosaic, mosaic, args.tile, args.tile, args.step, T,
                           ("YOLO" + args.variant) if args.variant.startswith('11') else ("YOLOv8" + args.variant), args.imgsz),
            "survey_config": args.config,
            "tiles": T, "tile_batch": args.batch, "parallelism": "tile-row bands x%d + NCCL all-gather of records" % n,
            "l2": "inputs larger than L2 (mosaic band >= 134 MB, activations > 1 GB per batch)",
            "score_thr": SCORE_THR, "iou_thr": IOU_THR}


def catalog_crc(src):
    """crc32 of the catalog bytes (cy_source records in catalog order): identical across GPU counts iff the catalogs are."""
    return "%08x" % (zlib.crc32(np.ascontiguousarray(src).view(np.uint8).tobytes()) & 0xffffffff)


DUMP_BYTES = 64 << 20      # cap on everything --dump-outputs writes


def dump_outputs(d, arrays):
    """Writes {name: array} as d/<name>.npy.  float32 / float64 arrays are written as they are, integer arrays as
    float64 (exact for int32)."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        np.save(os.path.join(d, name + '.npy'), a)


def catalog_arrays(src, nrec):
    """The catalog (cy_source array, catalog order) as one array per field plus the record count.  A catalog too large
    for DUMP_BYTES is cut to a fixed, seeded sample of its rows; `sources_row` then holds the rows kept."""
    out = {'records': np.array([nrec])}
    rows = DUMP_BYTES // (8 * (len(src.dtype.names) + 1))
    if len(src) > rows:
        keep = np.sort(np.random.default_rng(0).choice(len(src), rows, replace=False))
        src = src[keep]
        out['sources_row'] = keep
    out.update(('sources_' + f, src[f]) for f in src.dtype.names)
    return out


def match_fraction(got, want, thr):
    """Symmetric matched fraction of two catalog lists (dicts with x1,y1,x2,y2,class_id) at IoU >= thr, same class."""
    def iou(a, b):
        xl, yt = max(a['x1'], b['x1']), max(a['y1'], b['y1'])
        xr, yb = min(a['x2'], b['x2']), min(a['y2'], b['y2'])
        if xr <= xl or yb <= yt:
            return 0.0
        inter = (xr - xl) * (yb - yt)
        return inter / ((a['x2'] - a['x1']) * (a['y2'] - a['y1']) + (b['x2'] - b['x1']) * (b['y2'] - b['y1']) - inter)

    def one_way(A, Bs):
        used, m = set(), 0
        for a in A:
            best, bj = 0.0, -1
            for j, b in enumerate(Bs):
                if j in used or a['class_id'] != b['class_id'] or abs(a['x1'] - b['x1']) > 64 or abs(a['y1'] - b['y1']) > 64:
                    continue
                v = iou(a, b)
                if v > best:
                    best, bj = v, j
            if best >= thr:
                used.add(bj)
                m += 1
        return m / max(len(A), 1)
    if not got and not want:
        return 1.0
    return min(one_way(want, got), one_way(got, want))


def run_nms_stress(args):
    """--config 5 (BASELINE configs[4]): Detect decode -> threshold -> per-class NMS -> max_det -> un-letterbox
    (cy_postprocess) + per-tile IoU merge (cy_merge_tile) on 256 synthetic imgsz-1024 head-map tiles with ~10 k
    candidates each.  A step = one pass over the 256 tiles; HBM roofline: the head maps are read once (the K x K/64
    suppression bitmask of SURVEY §8d lives in shared memory, 512-box chunks)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import nms_stress
    from caesar_yolo_b200 import ops
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda:%d' % local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    hbm_peak, _, _, peak_kind = peaks()
    B, S, nc, conf = 256, 1024, 5, 0.05
    heads = nms_stress.rand_heads(B, S, S, nc, 42 + rank, -4.7, dev)     # independent tiles per rank (weak scaling)
    A = ops.num_anchors(S, S)
    _, _, lb = ops.letterbox_shape(args.tile, args.tile, S)
    lbd = ops.letterbox_array([lb] * B, dev)
    ncand = sum(int((torch.sigmoid(h[..., 64:64 + nc]).amax(-1) > conf).sum()) for h in heads) / float(B)
    need = int(ops.lib.cy_postprocess_scratch_bytes(B, S, S, ops.MAX_DET))
    scratch = torch.empty((need,), dtype=torch.uint8, device=dev)
    dets = torch.zeros((B, ops.MAX_DET, 6), dtype=torch.float32, device=dev)
    nd = torch.zeros((B,), dtype=torch.int32, device=dev)
    keep = torch.full((B, ops.MAX_DET), -1, dtype=torch.int32, device=dev)
    nkeep = torch.zeros((B,), dtype=torch.int32, device=dev)
    mstat = torch.zeros((B,), dtype=torch.int32, device=dev)

    def step():
        ops.postprocess(heads, B, S, S, nc, conf, IOU_THR, lbd, dev, scratch=scratch, dets=dets, ndets=nd)
        ops.merge_tile(dets, nd, conf, SOFT, HARD, keep_idx=keep, nkeep=nkeep, status=mstat)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(3, args.warmup)):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # rank 0's tiles: every rank draws its own head maps
        ndh, nkh = nd.cpu().numpy(), nkeep.cpu().numpy()
        dh, kh = dets.cpu().numpy(), keep.cpu().numpy()
        dump_outputs(args.dump_outputs, {
            'dets': np.concatenate([dh[i, :ndh[i]] for i in range(B)]), 'ndets': ndh,
            'keep_idx': np.concatenate([kh[i, :nkh[i]] for i in range(B)]), 'nkeep': nkh,
            'merge_status': mstat.cpu().numpy()})
    ms = float(t[0]) / args.steps
    # end to end: head maps from pinned host memory, kept indices back to the host
    hosts = [h.cpu().pin_memory() for h in heads]

    def step_e2e():
        for h, hh in zip(heads, hosts):
            h.copy_(hh, non_blocking=True)
        step()
        return keep.cpu(), nkeep.cpu()
    step_e2e()
    barrier()
    t0 = time.time()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_ms = (time.time() - t0) * 1e3 / args.steps
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    alg = (80 * A * 4 + ops.MAX_DET * 24) * B
    ach = alg / (ms * 1e-3) / 1e9
    line = {"metric": "tiles/s decode+NMS+merge", "value": B * world / (ms * 1e-3), "unit": "tiles/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[4]: %d tiles per GPU, imgsz %d (%d anchors), scoreThr %.2f, iou %.2f, "
                                   "nc 5, %.0f candidates per tile, synthetic head maps" % (B, S, A, conf, IOU_THR, ncand),
                       "survey_config": 5, "l2": "head maps 1.76 GB per step (> L2)"},
            "e2e": {"value": B * world / (e2e_ms * 1e-3), "unit": "tiles/s",
                    "h2d_bytes_per_step": int(sum(h.numel() * 4 for h in heads)),
                    "d2h_bytes_per_step": int(keep.numel() * 4 + nkeep.numel() * 4), "ms_per_step": e2e_ms},
            "gpu_launches": 4 * args.steps, "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "score_key_kernel + nms_tiles_kernel + merge_tile_kernel",
                         "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                         "peak_kind": peak_kind + " copy bandwidth", "traffic": None,
                         "algorithmic_bytes_per_launch": alg,
                         "note": "latency/IoU-test bound: the suppression bitmask stays in shared memory"},
            "dets_per_tile": float(nd.float().mean()), "kept_after_merge_per_tile": float(nkeep.float().mean())}
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs,
                                "outputs": "rank 0's %d tiles (the same head maps for any GPU count)" % B}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse()
    claim_stdout()
    if args.impl == 'reference':
        return run_reference(args)
    if args.config == 5:
        return run_nms_stress(args)
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda:%d' % local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    from caesar_yolo_b200 import catalog, ops, pipeline, weights as W
    hbm_peak, tf_sust, tf_burst, peak_kind = peaks()
    numa_node = pipeline.bind_host_to_device_numa(local) if world > 1 else None   # node-local pinned staging per rank

    img_native, host = make_mosaic_pinned(args)
    tiles = ops.generate_tiles(0, args.mosaic - 1, 0, args.mosaic - 1, args.tile, args.tile, args.step, args.step)
    T = len(tiles)
    w = W.make_random_weights(args.variant, 5, seed=0, cls_bias=CLS_BIAS.get(args.variant, -16.0))
    eng = pipeline.Engine(w, pipeline.make_pp_config(**PP_FLAGS), imgsz=args.imgsz, score_thr=SCORE_THR,
                          iou_thr=IOU_THR, thr_soft=SOFT, thr_hard=HARD, device=dev, batch_tiles=args.batch,
                          precision=args.precision)
    a, b = pipeline.split_tile_rows(tiles, world)[rank]
    y0b, y1b = int(tiles['ymin'][a:b].min()), int(tiles['ymax'][a:b].max())
    band_dev = host[y0b:y1b].to(dev)          # resident copy for the device-timed `value`
    my_ids = np.arange(a, b, dtype=np.int32)

    def step_resident():
        eng.begin(tiles)
        eng.process_tiles(band_dev, args.mosaic, True, 0, y0b, my_ids)
        return eng.exchange_and_merge(world)

    def step_e2e():
        return pipeline.run_image(eng, host, True, tiles, rank=rank, world=world, on_rank0_only=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        out = None
        for _ in range(k):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        wall = time.time() - t0
        barrier()
        t = torch.tensor([e0.elapsed_time(e1), wall * 1e3], dtype=torch.float64, device=dev)   # device time, wall time
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), out

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launches
    eng.stage_events = []                      # per-stage CUDA events recorded INSIDE the timed steps
    ms_dev, wall_ms, (src, nrec) = timed(step_resident, args.steps)
    stage_ms = {k: v / args.steps for k, v in eng.stage_times_ms().items()}
    eng.stage_events = None
    launches = eng.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, catalog_arrays(src, nrec))
    for _ in range(max(2, args.warmup - 1)):
        step_e2e()
    eng.stage_events = []
    ms_e2e, wall_e2e, (src2, _) = timed(step_e2e, args.steps)
    stage_ms_e2e = {k: v / args.steps for k, v in eng.stage_times_ms().items()}
    eng.stage_events = None

    # FITS FILE -> catalog: the mosaic is written to local disk once (outside the timer); every timed step reads this
    # rank's rows from the file into pinned staging buffers, uploads and processes them.
    file_info = None
    if not args.no_file:
        import tempfile
        from caesar_yolo_b200 import synth
        from caesar_yolo_b200.fits import FitsImage
        tmpd = tempfile.mkdtemp(prefix='cybench_')
        fpath = os.path.join(tmpd, 'mosaic_rank%d.fits' % rank)
        t0 = time.time()
        synth.write_fits_raw_be(fpath, host.numpy())
        t_write = time.time() - t0
        fimg = FitsImage(fpath)

        def step_file():
            return pipeline.run_image(eng, fimg, True, tiles, rank=rank, world=world, on_rank0_only=False)
        for _ in range(2):
            step_file()
        ms_f, wall_f, (src3, _) = timed(step_file, args.steps)
        file_ms = max(ms_f, wall_f) / args.steps
        # raw read rate of the same byte range with the same reader, nothing else running
        t0 = time.time()
        nbytes = pipeline.read_rows_benchmark(eng, fimg, y0b, y1b)
        t_read = time.time() - t0
        file_info = {"value": T / (file_ms * 1e-3), "unit": "tiles/s", "ms_per_step": file_ms,
                     "file_bytes_per_step": int(args.mosaic) * int(args.mosaic) * 4,
                     "host_read_GBps_alone": nbytes / t_read / 1e9,
                     "note": "file written once outside the timer (%.1f s) and served by the page cache afterwards; "
                             "read (preadv into pinned staging, %d reader threads) + H2D + compute overlapped; "
                             "catalog identical to `value`: %s" % (t_write, pipeline.READ_THREADS,
                                                                  bool(catalog_crc(src3) == catalog_crc(src)))}
        try:
            os.remove(fpath)
            os.rmdir(tmpd)
        except OSError:
            pass

    # The other 16-bit storage format on the same box, same workload (resident timing only): bf16 is the format
    # north_star names and draws less power per MMA than fp16 (the step sits at the board power cap), fp16 keeps three
    # more significand bits (parity).  Informational; the headline fields belong to the default format.
    alt = None
    if not args.no_alt:
        altp = 'bf16' if eng.model.precision == 'fp16' else 'fp16'
        eng2 = pipeline.Engine(w, pipeline.make_pp_config(**PP_FLAGS), imgsz=args.imgsz, score_thr=SCORE_THR,
                               iou_thr=IOU_THR, thr_soft=SOFT, thr_hard=HARD, device=dev, batch_tiles=args.batch,
                               precision=altp)

        def step_alt():
            eng2.begin(tiles)
            eng2.process_tiles(band_dev, args.mosaic, True, 0, y0b, my_ids)
            return eng2.exchange_and_merge(world)
        for _ in range(2):
            step_alt()
        eng2.stage_events = []
        ms2, _, (src_alt, _) = timed(step_alt, args.steps)
        st2 = {k: v / args.steps for k, v in eng2.stage_times_ms().items()}
        alt = {"dtype": altp, "value": T / (ms2 / args.steps * 1e-3), "unit": "tiles/s", "ms_per_step": ms2 / args.steps,
               "forward_ms_per_step": round(st2.get('forward', 0.0), 3), "sources": int(len(src_alt)),
               "note": "same box, same workload, mosaic resident; %d timed steps" % args.steps}
        del eng2

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    ms_step = ms_dev / args.steps
    value = T / (ms_step * 1e-3)
    e2e_ms = max(ms_e2e, wall_e2e) / args.steps     # host-facing call: wall clock covers the host side as well
    e2e_val = T / (e2e_ms * 1e-3)
    mpix = float(np.sum((tiles['xmax'] - tiles['xmin']).astype(np.int64) * (tiles['ymax'] - tiles['ymin'])) / 1e6)
    line = {"metric": "tiles/s FITS->catalog", "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": eng.model.precision, "data": "synthetic", "config": workload_config(args, world, T),
            "mpix_per_s": mpix / (ms_step * 1e-3), "sources": int(len(src)), "records": int(nrec),
            "catalog_crc32": catalog_crc(src), "catalog_crc32_e2e": catalog_crc(src2),
            "e2e": {"value": e2e_val, "unit": "tiles/s", "h2d_bytes_per_step": int(args.mosaic) * int(args.mosaic) * 4,
                    "d2h_bytes_per_step": int(len(src2)) * 32 * world, "ms_per_step": e2e_ms,
                    "mpix_per_s": mpix / (e2e_ms * 1e-3), "device_ms_per_step": ms_e2e / args.steps,
                    "wall_ms_per_step": wall_e2e / args.steps,
                    "stage_ms_per_step": {k: round(v, 3) for k, v in stage_ms_e2e.items()}},
            "gpu_launches": int(launches), "clocks": clocks,
            "stage_ms_per_step": {k: round(v, 3) for k, v in stage_ms.items()}}
    if file_info is not None:
        line["e2e_file"] = file_info
    if alt is not None:
        line["alt_precision"] = alt
    line["host_numa_node"] = numa_node       # node the rank-0 process (and its pinned staging) was bound to; None: not bound
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs,
                                "outputs": "merged catalog of the last timed step (the same for any GPU count)"}
    known = sum(stage_ms.get(k, 0.0) for k in ('preprocess', 'forward', 'decode_nms', 'merge_tile_records'))
    line["exchange_ms"] = round(stage_ms.get('exchange', 0.0), 3)
    line["unattributed_ms"] = round(ms_step - known - stage_ms.get('exchange', 0.0) - stage_ms.get('merge_global', 0.0), 3)

    # ---- rooflines, all from the CUDA events of the TIMED steps (rank 0's share of the tiles).
    Tr = b - a                                                    # tiles this rank processed per step
    Sh, Sw, _ = ops.letterbox_shape(args.tile, args.tile, args.imgsz)
    info = eng.model.info(min(args.batch, Tr), Sh, Sw)
    full = (tiles['xmax'] - tiles['xmin'] == args.tile) & (tiles['ymax'] - tiles['ymin'] == args.tile)
    # flops of this rank's tiles: full tiles at the planned shape, fragments scaled by area (edge tiles are letterboxed
    # to a proportionally smaller input)
    area = ((tiles['xmax'] - tiles['xmin']).astype(np.float64) * (tiles['ymax'] - tiles['ymin']))[a:b]
    flops_tile = info['flops'] / min(args.batch, Tr)
    fwd_flops = float(np.sum(area / float(args.tile * args.tile)) * flops_tile)
    fwd_ms = stage_ms.get('forward', 0.0)
    A = ops.num_anchors(Sh, Sw)
    pp_bytes = float(np.sum(area) * 4 + Tr * 2.0 * Sh * Sw * 4)   # read tile once + write bf16 NHWC (Cpad = 4) once
    dec_bytes = Tr * (80.0 * A * 4 + ops.MAX_DET * 24)            # head maps (fp32, 80 floats per anchor) + dets
    mt_bytes = Tr * (ops.MAX_DET * 24 + ops.MAX_DET * 4 + ops.MAX_DET * 32)
    mg_bytes = float(nrec) * 64.0

    def hbm_entry(ms, nbytes, kernels):
        ach = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        return {"bound": "hbm", "kernels": kernels, "ms_per_step": round(ms, 4), "algorithmic_bytes_per_step": nbytes,
                "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak}
    line["roofline_by_stage"] = {
        "preprocess": hbm_entry(stage_ms.get('preprocess', 0.0), pp_bytes, eng.pp_kernels()),
        "forward": {"bound": "tensor", "kernels": "conv_igemm_kernel x%d + stem / pool / upsample per batch" % int(info['nconv']),
                    "ms_per_step": round(fwd_ms, 4), "algorithmic_flops_per_step": fwd_flops,
                    "achieved": fwd_flops / (fwd_ms * 1e-3) / 1e12 if fwd_ms > 0 else 0.0, "peak": tf_sust,
                    "unit": "TFLOP/s", "frac": (fwd_flops / (fwd_ms * 1e-3) / 1e12 / tf_sust) if fwd_ms > 0 else 0.0},
        "decode_nms": hbm_entry(stage_ms.get('decode_nms', 0.0), dec_bytes, "score_key_kernel + nms_tiles_kernel"),
        "merge_tile_records": hbm_entry(stage_ms.get('merge_tile_records', 0.0), mt_bytes,
                                        "merge_tile_kernel + make_records_kernel"),
        "merge_global": hbm_entry(stage_ms.get('merge_global', 0.0), mg_bytes, "merge_global.cu kernels"),
        "peak_kind": "%s: HBM copy bandwidth / sustained bf16 cuBLAS (kernels timed inside a long step)" % peak_kind,
        "timing": "CUDA events around each stage inside the timed steps (stream order), rank 0, divided by the step count"}

    # ---- roofline of the dominant kernel (the tcgen05 implicit-GEMM conv): the whole forward stage of the TIMED steps
    # (conv launches + the stem / pool / upsample kernels, 3-4 % of it) against the conv FLOPs — a lower bound on the
    # conv kernel's own rate; the per-layer profile below (one extra batch, outside the timed region) splits it.
    nconv_launches = int(info['nconv']) * int(np.ceil(Tr / float(args.batch)))
    ach = fwd_flops / (fwd_ms * 1e-3) / 1e12 if fwd_ms > 0 else 0.0
    line["roofline"] = {"bound": "tensor", "kernel": "conv_igemm_kernel (tcgen05 implicit GEMM, %d launches per batch of %d tiles)" % (int(info['nconv']), args.batch),
                        "achieved": ach, "peak": tf_sust, "unit": "TFLOP/s", "frac": ach / tf_sust,
                        "peak_kind": "%s sustained bf16 cuBLAS (kernel timed inside a long step)" % peak_kind,
                        "measured": "forward-stage CUDA events of the timed steps (includes the non-conv kernels of the forward)",
                        "traffic": None, "avg_launch_us": fwd_ms * 1e3 / max(nconv_launches, 1),
                        "algorithmic_flops_per_launch": fwd_flops / max(nconv_launches, 1)}
    if not args.no_profile:
        x = torch.rand((args.batch, Sh, Sw, 4), device=dev).to(eng.model.dtype)
        prof = eng.model.profile(x)
        prof = eng.model.profile(x)
        conv = [(n_, ms, fl) for (n_, ms, fl) in prof if fl > 0 and n_ != 'model.0']
        conv_ms = sum(p[1] for p in conv)
        conv_fl = sum(p[2] for p in conv)
        tot_ms = sum(p[1] for p in prof)
        line["roofline"]["conv_only_profile"] = {
            "achieved": conv_fl / (conv_ms * 1e-3) / 1e12, "frac": conv_fl / (conv_ms * 1e-3) / 1e12 / tf_sust,
            "conv_share_of_forward": conv_ms / tot_ms, "note": "per-op CUDA events of one extra batch (random input) after the timed region"}
        try:
            if args.variant != 'l' or args.imgsz != 640 or args.tile != 512:
                raise ValueError('the committed ncu capture is of the yolov8l / 512 / 640 workload')
            tj = json.load(open(os.path.join(ROOT, 'profiles', 'conv_traffic.json')))
            line["roofline"]["traffic"] = (tj["dram_read_bytes"] + tj["dram_write_bytes"]) / tj["conv_launches"] * (
                args.batch / float(tj["tiles"]))
            line["roofline"]["traffic_source"] = tj["source"]
            line["roofline"]["tensor_pipe_active_pct_ncu"] = tj.get("tensor_pipe_active_pct_time_weighted")
        except Exception:
            pass
        ab, nconv = eng.model.conv_bytes(args.batch, Sh, Sw)
        line["roofline"]["algorithmic_bytes_per_launch"] = ab / max(nconv, 1)
        slow = sorted(prof, key=lambda p: -p[1])[:8]
        line["roofline"]["top_ops"] = [{"op": n_, "ms": round(ms, 4), "tflops": round(fl / (ms * 1e-3) / 1e12, 1) if ms > 0 else 0} for n_, ms, fl in slow]

    if not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        n = sample_side(args)
        sub = np.ascontiguousarray(img_native[:n, :n])
        v, dt, nt, ocat = cpu_reference(args, sub, threads, keep_catalog=True)
        line["cpu_baseline"] = {"value": v, "unit": "tiles/s", "cores": threads, "kind": "port",
                                "sample": "%d tiles (top-left %dx%d sub-mosaic of the benchmark mosaic), oracle SFinder.run_parallel FITS->catalog in %.1f s, torch CPU fp32 batch 1, logging silenced" % (nt, n, n, dt)}
        # parity of the benchmarked configuration: the SAME sub-mosaic through this engine (same weights, thresholds,
        # batch plan) against the oracle catalog just computed
        stiles = ops.generate_tiles(0, n - 1, 0, n - 1, args.tile, args.tile, args.step, args.step)
        sub_be = torch.from_numpy(sub.astype('>f4').view(np.int32).copy())
        gsrc, _ = pipeline.run_image(eng, sub_be, True, stiles, rank=0, world=1)
        gcat = catalog.sources_to_dicts(gsrc, eng.names)
        line["parity_check"] = {"sample": "%d tiles, same weights / thresholds as the timed run" % len(stiles),
                                "oracle": "fp32 CPU port (the %s storage of the conv stack is the only intended difference)" % eng.model.precision,
                                "sources_gpu": len(gcat), "sources_oracle": len(ocat),
                                "matched_iou0.9": match_fraction(gcat, ocat, 0.9),
                                "matched_iou0.5": match_fraction(gcat, ocat, 0.5),
                                "catalog_crc32_gpu_sample": catalog_crc(gsrc)}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
