"""Thin Python handles on the C-ABI stage kernels (torch used only for device memory + streams).
Every function here calls libcaesar_b200.so; there is no CPU or torch fallback."""
import ctypes
import os

import numpy as np
import torch

from . import _capi
from ._capi import (CaesarB200Error, PPChain, PPConfig, Letterbox, c_int, c_float, c_double, c_i64, c_void_p, check, cur_stream,
                    lib, ptr)

MAX_DET = 300          # ultralytics non_max_suppression max_det
DET_STRIDE = 304       # per-tile detection slots (>= MAX_DET, <= 320)
HEAD_C = 80            # per-anchor head record (64 DFL logits + up to 16 class logits)

TILE_DTYPE = np.dtype([('xmin', '<i4'), ('xmax', '<i4'), ('ymin', '<i4'), ('ymax', '<i4')])
REC_DTYPE = np.dtype([('x1', '<f4'), ('y1', '<f4'), ('x2', '<f4'), ('y2', '<f4'), ('score', '<f4'), ('cls', '<i4'),
                      ('tile_id', '<i4'), ('flags', '<i4')])
SRC_DTYPE = np.dtype([('x1', '<f4'), ('y1', '<f4'), ('x2', '<f4'), ('y2', '<f4'), ('score', '<f4'), ('cls', '<i4'),
                      ('flags', '<i4'), ('tile_id', '<i4')])


def _np_ptr(a):
    return c_void_p(a.ctypes.data)


# ------------------------------------------------------------------------------------------------ tiling (host)

def generate_tiles(xmin, xmax, ymin, ymax, tile_x, tile_y, step_x, step_y):
    """utils.generate_tiles (caesar_yolo/utils.py:622-697) -> structured array (xmin, xmax_excl, ymin, ymax_excl)
    or None on invalid arguments (the reference returns None and logs)."""
    n = c_int(0)
    args = (c_int(xmin), c_int(xmax), c_int(ymin), c_int(ymax), c_int(tile_x), c_int(tile_y), c_double(step_x),
            c_double(step_y))
    if lib.cy_generate_tiles(*args, c_void_p(0), c_int(0), ctypes.byref(n)) != 0:
        return None
    tiles = np.zeros(n.value, dtype=TILE_DTYPE)
    check(lib.cy_generate_tiles(*args, _np_ptr(tiles), c_int(n.value), ctypes.byref(n)))
    return tiles


def tile_neighbors(tiles):
    """Neighbour CSR (nb_off[T+1], nb_idx) of SFinder.create_tile_tasks (inference.py:1034-1071)."""
    T = len(tiles)
    off = np.zeros(T + 1, dtype=np.int32)
    total = c_int(0)
    check(lib.cy_tile_neighbors(_np_ptr(tiles), c_int(T), _np_ptr(off), c_void_p(0), c_int(0), ctypes.byref(total)))
    idx = np.zeros(max(total.value, 1), dtype=np.int32)
    check(lib.cy_tile_neighbors(_np_ptr(tiles), c_int(T), _np_ptr(off), _np_ptr(idx), c_int(total.value),
                                ctypes.byref(total)))
    return off, idx[:total.value]


# ------------------------------------------------------------------------------------------------ preprocessing

def letterbox_shape(Ty, Tx, imgsz):
    sh, sw = c_int(0), c_int(0)
    lb = Letterbox()
    check(lib.cy_letterbox_shape(c_int(Ty), c_int(Tx), c_int(imgsz), ctypes.byref(sh), ctypes.byref(sw),
                                 ctypes.byref(lb)))
    return sh.value, sw.value, lb


# 16-bit storage format of weights / activations.  fp16 and bf16 run on the same tcgen05 kind::f16 instruction at the same
# rate with fp32 accumulation; fp16 keeps 11 significand bits instead of 8, which is what decides how closely the
# catalogs follow the reference's fp32 arithmetic (DESIGN.md §7: matched fraction 0.986 vs 0.919 on the same mosaic;
# the reference's own TF32 GPU path reaches 0.993), and it is the type ultralytics' `half=True` uses.
DEFAULT_PRECISION = os.environ.get('CY_PRECISION', 'fp16')


def chain_from_config(cfg):
    """cy_pp_config (run.py's option set) -> cy_pp_chain (the stage list in run.py's order)."""
    ch = PPChain()
    check(lib.cy_pp_chain_from_config(ctypes.byref(cfg), ctypes.byref(ch)))
    return ch


def validate_chain(ch):
    check(lib.cy_pp_chain_validate(ctypes.byref(ch)))
    return ch


def storage_dtype(precision):
    """torch dtype of the 16-bit storage format: 'fp16' or 'bf16' (None: DEFAULT_PRECISION)."""
    if precision is None:
        precision = DEFAULT_PRECISION
    if precision in ('bf16', 0, False):
        return torch.bfloat16
    if precision in ('fp16', 'f16', 'half', 1, True):
        return torch.float16
    raise ValueError("precision must be 'bf16' or 'fp16' (got %r)" % (precision,))


def preprocess(cfg, img, row_stride, big_endian, tile_x0, tile_y0, Ty, Tx, imgsz, want_f32=False, scratch=None,
               chain_out=None, model_in=None, status=None, want_chain=True):
    """cy_preprocess.  img: device tensor (any dtype of 4-byte elements); tile_x0/y0: int32 device tensors [B].
    Returns (chain_out [B,Ty,Tx,3] f32 or None, model_in [B,Sh,Sw,4] bf16 / fp16 (cfg.out_f16), model_in_f32 or None,
    status [B] i32).  want_chain=False skips the fp32 chain image (the production path: it only exists for parity)."""
    B = tile_x0.numel()
    dev = img.device
    is_chain = isinstance(cfg, PPChain)     # a general stage list (cy_preprocess_chain) or run.py's option set
    Sh, Sw, _ = letterbox_shape(Ty, Tx, imgsz)
    if chain_out is None and want_chain:
        chain_out = torch.empty((B, Ty, Tx, 3), dtype=torch.float32, device=dev)
    if model_in is None:
        model_in = torch.empty((B, Sh, Sw, 4), dtype=torch.float16 if cfg.out_f16 else torch.bfloat16, device=dev)
    f32 = torch.empty((B, 3, Sh, Sw), dtype=torch.float32, device=dev) if want_f32 else None
    if status is None:
        status = torch.empty((B,), dtype=torch.int32, device=dev)
    size_fn = lib.cy_preprocess_chain_scratch_bytes if is_chain else lib.cy_preprocess_scratch_bytes
    need = int(size_fn(ctypes.byref(cfg), c_int(B), c_int(Ty), c_int(Tx)))
    if need == 0:
        raise CaesarB200Error("invalid preprocessing chain / tile shape: %s" % lib.cy_last_error().decode())
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty((need,), dtype=torch.uint8, device=dev)
    fn = lib.cy_preprocess_chain if is_chain else lib.cy_preprocess
    check(fn(ctypes.byref(cfg), ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0),
             ptr(tile_x0), ptr(tile_y0), c_int(B), c_int(Ty), c_int(Tx), c_int(imgsz), ptr(chain_out),
             ptr(model_in), ptr(f32), ptr(status), ptr(scratch), cur_stream()))
    return chain_out, model_in, f32, status


def letterbox_resize(chain, imgsz, want_f32=False, dtype=torch.bfloat16):
    """chain: [B,Ty,Tx,3] f32 device -> model_in [B,Sh,Sw,4] bf16 / fp16 (+ optional f32 NCHW)."""
    B, Ty, Tx, _ = chain.shape
    Sh, Sw, _ = letterbox_shape(Ty, Tx, imgsz)
    model_in = torch.empty((B, Sh, Sw, 4), dtype=dtype, device=chain.device)
    f32 = torch.empty((B, 3, Sh, Sw), dtype=torch.float32, device=chain.device) if want_f32 else None
    check(lib.cy_letterbox_resize_fmt(ptr(chain), c_int(B), c_int(Ty), c_int(Tx), c_int(imgsz), ptr(model_in),
                                      ptr(f32), c_int(1 if dtype == torch.float16 else 0), cur_stream()))
    return model_in, f32


# ------------------------------------------------------------------------------------------------ conv primitive

def conv_block_n(cout):
    return int(lib.cy_conv_block_n(c_int(cout)))


def pack_conv_weight(w_oihw, bias, device):
    """[Cout,Cin,kh,kw] float/bf16 (BN already folded) -> device bf16 [cout_pad, kh*kw*Cin] + fp32 bias[cout_pad]."""
    cout, cin, kh, kw = w_oihw.shape
    bn = conv_block_n(cout)
    cout_pad = (cout + bn - 1) // bn * bn
    wp = torch.zeros(cout_pad, kh * kw * cin, dtype=torch.bfloat16)
    wp[:cout] = w_oihw.permute(0, 2, 3, 1).reshape(cout, -1).to(torch.bfloat16)
    bp = torch.zeros(cout_pad, dtype=torch.float32)
    if bias is not None:
        bp[:cout] = bias.float()
    return wp.to(device), bp.to(device)


def conv2d_nhwc(x, in_coff, cin, wp, bp, cout, k, s, out, out_coff, act=True, res=None, res_coff=0):
    B, H, W, in_ctot = x.shape
    check(lib.cy_conv2d_nhwc(ptr(x), c_int(B), c_int(H), c_int(W), c_int(in_ctot), c_int(in_coff), c_int(cin),
                             ptr(wp), ptr(bp), c_int(cout), c_int(wp.shape[0]), c_int(k), c_int(s), ptr(out),
                             c_int(out.shape[-1]), c_int(out_coff), c_int(1 if out.dtype == torch.float32 else 0),
                             ptr(res), c_int(res.shape[-1] if res is not None else 0), c_int(res_coff),
                             c_int(1 if act else 0), cur_stream()))


def stem_conv(x, w_oihw, bias, act=1):
    """Fused stem (cy_stem_conv_nhwc4): x [B,H,W,4] bf16 on the device, w [cout,3,3,3] / bias [cout] host fp32 (BN folded)
    -> [B,H/2,W/2,cout] bf16."""
    B, H, W, C = x.shape
    assert C == 4 and x.dtype == torch.bfloat16 and x.is_contiguous()
    cout = int(w_oihw.shape[0])
    w = np.ascontiguousarray(w_oihw.detach().cpu().float().numpy())
    b = np.ascontiguousarray(bias.detach().cpu().float().numpy())
    out = torch.empty((B, H // 2, W // 2, cout), dtype=torch.bfloat16, device=x.device)
    check(lib.cy_stem_conv_nhwc4(ptr(x), c_int(B), c_int(H), c_int(W), _np_ptr(w), _np_ptr(b), c_int(cout),
                                 c_int(int(act)), ptr(out), cur_stream()))
    return out


# ------------------------------------------------------------------------------------------------ model

class DeviceModel(object):
    """YOLOv8 DetectionModel resident on the current CUDA device (cy_model_*)."""

    def __init__(self, weights, precision=None):
        self.variant = weights['variant']
        self.nc = int(weights['nc'])
        self.names = dict(weights['names'])
        self.dtype = storage_dtype(precision)
        self.precision = 'fp16' if self.dtype == torch.float16 else 'bf16'
        h = c_void_p(0)
        check(lib.cy_model_create(self.variant.encode(), c_int(self.nc), ctypes.byref(h)))
        self._h = h
        check(lib.cy_model_set_precision(self._h, c_int(1 if self.dtype == torch.float16 else 0)))
        for k, v in weights['state_dict'].items():
            if '.dfl.' in k:
                continue
            a = np.ascontiguousarray(v.detach().cpu().float().numpy())
            check(lib.cy_model_set_tensor(self._h, k.encode(), _np_ptr(a), c_i64(a.size)))
        check(lib.cy_model_finalize(self._h))

    def forward(self, x):
        """x: [B,Sh,Sw,4] NHWC in the model's storage format (bf16 / fp16) -> three raw head maps [B,h,w,80] f32 (views
        of model-owned buffers)."""
        B, Sh, Sw, C = x.shape
        if x.dtype != self.dtype:
            raise CaesarB200Error("model input is %s but the model stores %s" % (x.dtype, self.dtype))
        assert C == 4 and x.is_contiguous()
        heads = (c_void_p * 3)()
        check(lib.cy_model_forward(self._h, ptr(x), c_int(B), c_int(Sh), c_int(Sw), heads, cur_stream()))
        return [int(heads[l]) for l in range(3)]

    def forward_tensors(self, x):
        """Like forward() but copies the head maps into fresh torch tensors (tests)."""
        B, Sh, Sw, _ = x.shape
        ptrs = self.forward(x)
        outs = []
        for l, p in enumerate(ptrs):
            s = 8 << l
            t = torch.empty((B, Sh // s, Sw // s, HEAD_C), dtype=torch.float32, device=x.device)
            _capi.cuda_memcpy_d2d(t.data_ptr(), p, t.numel() * 4)
            outs.append(t)
        return outs

    def info(self, B, Sh, Sw):
        a = (c_double * 8)()
        check(lib.cy_model_info(self._h, c_int(B), c_int(Sh), c_int(Sw), a))
        keys = ('nparams', 'flops', 'launches', 'act_bytes', 'c3', 'c4', 'c5', 'nconv')
        return dict(zip(keys, [float(v) for v in a]))

    def plan_summary(self, B, Sh, Sw):
        """What the planner chose for this shape: launches by kind (cy_model_plan_summary)."""
        a = (c_int * 8)()
        check(lib.cy_model_plan_summary(self._h, c_int(B), c_int(Sh), c_int(Sw), a))
        keys = ('conv_launches', 'pair_launches', 'mode0_launches', 'mode1_launches', 'mode2_launches',
                'mode3_launches', 'wide_launches', 'two_half_launches')
        return dict(zip(keys, [int(v) for v in a]))

    def conv_bytes(self, B, Sh, Sw):
        """(algorithmic HBM bytes of all conv launches of one forward, number of conv launches)."""
        b = c_double(0.0)
        n = c_int(0)
        check(lib.cy_model_conv_bytes(self._h, c_int(B), c_int(Sh), c_int(Sw), ctypes.byref(b), ctypes.byref(n)))
        return float(b.value), int(n.value)

    def profile(self, x):
        B, Sh, Sw, _ = x.shape
        cap = 512
        names = (ctypes.c_char_p * cap)()
        ms = (c_float * cap)()
        fl = (c_double * cap)()
        n = c_int(0)
        check(lib.cy_model_profile(self._h, ptr(x), c_int(B), c_int(Sh), c_int(Sw), c_int(cap), names, ms, fl,
                                   ctypes.byref(n), cur_stream()))
        return [(names[i].decode(), float(ms[i]), float(fl[i])) for i in range(min(n.value, cap))]

    def __del__(self):
        try:
            if self._h:
                lib.cy_model_destroy(self._h)
                self._h = c_void_p(0)
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------ detect / NMS

def num_anchors(Sh, Sw):
    return int(lib.cy_num_anchors(c_int(Sh), c_int(Sw)))


def decode_pred(heads, B, Sh, Sw, nc, device):
    A = num_anchors(Sh, Sw)
    pred = torch.empty((B, 4 + nc, A), dtype=torch.float32, device=device)
    hp = [c_void_p(h) if isinstance(h, int) else ptr(h) for h in heads]
    check(lib.cy_decode_pred(hp[0], hp[1], hp[2], c_int(B), c_int(Sh), c_int(Sw), c_int(nc), ptr(pred), cur_stream()))
    return pred


def letterbox_array(lbs, device):
    """list of Letterbox -> device byte tensor holding cy_letterbox[B]."""
    arr = (Letterbox * len(lbs))(*lbs)
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
    return host.to(device)


def postprocess(heads, B, Sh, Sw, nc, conf, iou, lb_dev, device, max_det=MAX_DET, scratch=None, dets=None, ndets=None):
    need = int(lib.cy_postprocess_scratch_bytes(c_int(B), c_int(Sh), c_int(Sw), c_int(max_det)))
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty((need,), dtype=torch.uint8, device=device)
    if dets is None:
        dets = torch.zeros((B, max_det, 6), dtype=torch.float32, device=device)
    if ndets is None:
        ndets = torch.zeros((B,), dtype=torch.int32, device=device)
    hp = [c_void_p(h) if isinstance(h, int) else ptr(h) for h in heads]
    check(lib.cy_postprocess(hp[0], hp[1], hp[2], c_int(B), c_int(Sh), c_int(Sw), c_int(nc), c_float(conf),
                             c_float(iou), c_int(max_det), ptr(lb_dev), ptr(dets), ptr(ndets), ptr(scratch),
                             cur_stream()))
    return dets, ndets


def nms_batched(boxes, scores, iou_thr, counts=None, max_keep=0):
    """== torchvision.ops.nms per segment.  boxes [B,N,4] f32, scores [B,N] f32 -> keep [B,N] i64, nkeep [B] i32."""
    B, N, _ = boxes.shape
    dev = boxes.device
    need = int(lib.cy_nms_scratch_bytes(c_int(B), c_int(N)))
    scratch = torch.empty((need,), dtype=torch.uint8, device=dev)
    keep = torch.full((B, N), -1, dtype=torch.int64, device=dev)
    nkeep = torch.zeros((B,), dtype=torch.int32, device=dev)
    check(lib.cy_nms_batched(ptr(boxes), ptr(scores), ptr(counts), c_int(B), c_int(N), c_double(iou_thr),
                             c_int(max_keep), ptr(keep), ptr(nkeep), ptr(scratch), cur_stream()))
    return keep, nkeep


# ------------------------------------------------------------------------------------------------ merges

def merge_tile(dets, ndets, thr_score, thr_soft, thr_hard, keep_idx=None, nkeep=None, status=None, pre_status=None):
    B, stride, _ = dets.shape
    dev = dets.device
    if keep_idx is None:
        keep_idx = torch.full((B, stride), -1, dtype=torch.int32, device=dev)
    if nkeep is None:
        nkeep = torch.zeros((B,), dtype=torch.int32, device=dev)
    if status is None:
        status = torch.zeros((B,), dtype=torch.int32, device=dev)
    check(lib.cy_merge_tile(ptr(dets), ptr(ndets), c_int(B), c_int(stride), c_float(thr_score), c_float(thr_soft),
                            c_float(thr_hard), ptr(pre_status), ptr(keep_idx), ptr(nkeep), ptr(status), cur_stream()))
    return keep_idx, nkeep, status


def make_records(dets, keep_idx, nkeep, status, tiles_dev, tile_ids, recs, nrec):
    B, stride, _ = dets.shape
    check(lib.cy_make_records(ptr(dets), ptr(keep_idx), ptr(nkeep), ptr(status), c_int(stride), ptr(tiles_dev),
                              ptr(tile_ids), c_int(B), ptr(recs), ptr(nrec), cur_stream()))


def compact_records(slots, counts, T, slot_stride, out, total, scratch=None):
    dev = slots.device
    need = int(lib.cy_compact_scratch_bytes(c_int(T)))
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty((need,), dtype=torch.uint8, device=dev)
    check(lib.cy_compact_records(ptr(slots), ptr(counts), c_int(T), c_int(slot_stride), ptr(out), ptr(total),
                                 ptr(scratch), cur_stream()))


def merge_global(recs, n, tiles_dev, T, nb_off_dev, nb_idx_dev, out=None):
    """recs: uint8 device tensor of n cy_det_record (tile-id major).  Returns numpy structured array of cy_source."""
    dev = recs.device
    if out is None:
        out = torch.empty((max(n, 1) * SRC_DTYPE.itemsize,), dtype=torch.uint8, device=dev)
    nout = torch.zeros((1,), dtype=torch.int64, device=dev)
    check(lib.cy_merge_global(ptr(recs), c_int(n), ptr(tiles_dev), c_int(T), ptr(nb_off_dev), ptr(nb_idx_dev),
                              ptr(out), ptr(nout), cur_stream()))
    k = int(nout.item())
    return out[:k * SRC_DTYPE.itemsize].cpu().numpy().view(SRC_DTYPE)


# ------------------------------------------------------------------------------------------------ measurements

PARTIAL_BYTES = ctypes.sizeof(_capi.SrcPartial)
MEAS_DTYPE = np.dtype([('npix', '<i8'), ('sum', '<f8'), ('peak', '<f8'), ('peak_x', '<f8'), ('peak_y', '<f8'),
                       ('xc', '<f8'), ('yc', '<f8'), ('a', '<f8'), ('b', '<f8'), ('theta', '<f8')])
PARTIAL_DTYPE = np.dtype([('npix', '<i8'), ('peak_idx', '<i8'), ('peak', '<f8'), ('sum', '<f8'), ('sw', '<f8'),
                          ('swx', '<f8'), ('swy', '<f8'), ('swxx', '<f8'), ('swyy', '<f8'), ('swxy', '<f8')])
assert MEAS_DTYPE.itemsize == ctypes.sizeof(_capi.SrcMeas) and PARTIAL_DTYPE.itemsize == PARTIAL_BYTES


def measure_sources(img, row_stride, big_endian, row0, ncols, src_dev, nsrc, row_begin, row_end, out=None):
    """cy_measure_sources.  img: device tensor of 4-byte pixels whose first element is (row0, column 0); src_dev: uint8
    device tensor of nsrc cy_source.  Returns the partials as a uint8 device tensor [nsrc * 80] (synchronises)."""
    if out is None:
        out = torch.empty((max(nsrc, 1) * PARTIAL_BYTES,), dtype=torch.uint8, device=src_dev.device)
    check(lib.cy_measure_sources(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0),
                                 c_int(ncols), ptr(src_dev), c_int(nsrc), c_int(row_begin), c_int(row_end), ptr(out),
                                 cur_stream()))
    return out[:nsrc * PARTIAL_BYTES]


def measure_combine(partials, world, src_dev, nsrc, ncols, out=None):
    """cy_measure_combine: partials [world * nsrc * 80] uint8 device (rank-major) -> uint8 device tensor of nsrc
    cy_src_meas."""
    if out is None:
        out = torch.empty((max(nsrc, 1) * MEAS_DTYPE.itemsize,), dtype=torch.uint8, device=partials.device)
    check(lib.cy_measure_combine(ptr(partials), c_int(world), ptr(src_dev), c_int(nsrc), c_int(ncols), ptr(out),
                                 cur_stream()))
    return out[:nsrc * MEAS_DTYPE.itemsize]


NOISE_PARTIAL_BYTES = ctypes.sizeof(_capi.NoisePartial)
NOISE_DTYPE = np.dtype([('lo', '<f8'), ('hi', '<f8'), ('c', '<f8'), ('bkg', '<f8'), ('rms', '<f8'), ('nbkg', '<i8'),
                        ('iters', '<i4'), ('done', '<i4')])
NOISE_PARTIAL_DTYPE = np.dtype([('n', '<i8'), ('s1', '<f8'), ('s2', '<f8')])
NOISE_MAX_PASSES = 6   # pass 0 and up to 5 clipping iterations
assert NOISE_DTYPE.itemsize == ctypes.sizeof(_capi.NoiseState) and NOISE_PARTIAL_DTYPE.itemsize == NOISE_PARTIAL_BYTES


def noise_init(src_dev, nsrc, ncols, row_begin, row_end, frame, state, unit_off):
    """cy_noise_init.  state: uint8 device tensor of >= nsrc cy_noise_state; unit_off: int64 device tensor of >= nsrc + 1
    elements.  Returns the number of work units (synchronises)."""
    units = c_i64(0)
    check(lib.cy_noise_init(ptr(src_dev), c_int(nsrc), c_int(ncols), c_int(row_begin), c_int(row_end), c_int(frame),
                            ptr(state), ptr(unit_off), ctypes.byref(units), cur_stream()))
    return units.value


def noise_pass(img, row_stride, big_endian, row0, ncols, src_dev, nsrc, row_begin, row_end, frame, unit_off, units,
               state, out):
    """cy_noise_pass: one clipping pass over this range's rows -> out, uint8 device tensor of nsrc cy_noise_partial."""
    check(lib.cy_noise_pass(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(ncols),
                            ptr(src_dev), c_int(nsrc), c_int(row_begin), c_int(row_end), c_int(frame), ptr(unit_off),
                            c_i64(units), ptr(state), ptr(out), cur_stream()))
    return out


def noise_pass_masked(img, row_stride, big_endian, row0, ncols, src_dev, nsrc, row_begin, row_end, frame, unit_off,
                      units, state, out, mask):
    """cy_noise_pass_masked: noise_pass with the frame pixels in the source mask (source_mask of the same sources,
    ncols and rows) masked."""
    check(lib.cy_noise_pass_masked(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0),
                                   c_int(ncols), ptr(src_dev), c_int(nsrc), c_int(row_begin), c_int(row_end),
                                   c_int(frame), ptr(unit_off), c_i64(units), ptr(state), ptr(out), ptr(mask),
                                   cur_stream()))
    return out


def source_mask_words(ncols):
    """uint32 words per row of a source mask of ncols columns."""
    return (ncols + 31) // 32


def source_mask(src_dev, nsrc, ncols, row_begin, row_end, out=None):
    """cy_source_mask: bit mask of the union of the catalog boxes over columns [0, ncols) and rows [row_begin, row_end)
    -> int32 device tensor [row_end - row_begin, source_mask_words(ncols)] (bit x & 31 of word x >> 5 of row
    y - row_begin: pixel (x, y) lies in a box; synchronises)."""
    shape = (row_end - row_begin, source_mask_words(ncols))
    if out is None:
        out = torch.empty(shape, dtype=torch.int32, device=src_dev.device)
    check(lib.cy_source_mask(ptr(src_dev), c_int(nsrc), c_int(ncols), c_int(row_begin), c_int(row_end), ptr(out),
                             cur_stream()))
    return out


def noise_update(partials, world, nsrc, state):
    """cy_noise_update: partials [world * nsrc * 24] uint8 device (rank-major) -> state advanced by one pass.  Returns
    the number of sources still active (synchronises)."""
    active = c_int(0)
    check(lib.cy_noise_update(ptr(partials), c_int(world), c_int(nsrc), ptr(state), ctypes.byref(active),
                              cur_stream()))
    return active.value


BKG_ESTIMATORS = ('mean', 'median')
SELECT_BYTES = ctypes.sizeof(_capi.SelectState)
SELECT_SLOTS = 512    # uint32 histogram slots per source or node: 256 bins for each of the two middle ranks
SELECT_ROUNDS = 4     # 8-bit digit rounds of the median select per clipping pass


def noise_pass_median(img, row_stride, big_endian, row0, ncols, src_dev, nsrc, row_begin, row_end, frame, unit_off,
                      units, state, sel, rnd, out, hist, mask=None):
    """cy_noise_pass_median[_masked]: round rnd of a median pass over this range's rows -> hist (int32 device tensor of
    nsrc * SELECT_SLOTS uint32 counts) and, in round 0, out (as noise_pass).  mask: source_mask, or None."""
    args = [ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(ncols), ptr(src_dev),
            c_int(nsrc), c_int(row_begin), c_int(row_end), c_int(frame), ptr(unit_off), c_i64(units), ptr(state),
            ptr(sel), c_int(rnd), ptr(out), ptr(hist)]
    if mask is None:
        check(lib.cy_noise_pass_median(*args, cur_stream()))
    else:
        check(lib.cy_noise_pass_median_masked(*args, ptr(mask), cur_stream()))


def bkg_grid_pass_median(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid, unit_off,
                         units, state, sel, rnd, out, hist, mask=None, mask_ncols=0, mask_col0=0):
    """cy_bkg_grid_pass_median[_masked]: round rnd of a median pass of the grid nodes -> hist (Nx * Ny * SELECT_SLOTS
    counts) and, in round 0, out (as bkg_grid_pass).  mask: as for bkg_grid_pass_masked, or None."""
    args = [ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(ncols), c_int(R0),
            c_int(R1), c_int(row_begin), c_int(row_end), c_int(box), c_int(grid), ptr(unit_off), c_i64(units),
            ptr(state), ptr(sel), c_int(rnd), ptr(out), ptr(hist)]
    if mask is None:
        check(lib.cy_bkg_grid_pass_median(*args, cur_stream()))
    else:
        check(lib.cy_bkg_grid_pass_median_masked(*args, ptr(mask), c_int(mask_ncols), c_int(mask_col0), cur_stream()))


def median_update(partials, world, hist, n, state, sel, rnd):
    """cy_median_update: round rnd of a median pass, with hist summed over the ranks (and, in round 0, the partials
    [world * n * 24] gathered in rank order).  Returns the number still active after the last round (synchronises),
    None after the others (no synchronisation)."""
    if rnd < SELECT_ROUNDS - 1:
        check(lib.cy_median_update(ptr(partials), c_int(world), ptr(hist), c_int(n), ptr(state), ptr(sel), c_int(rnd),
                                   None, cur_stream()))
        return None
    active = c_int(0)
    check(lib.cy_median_update(ptr(partials), c_int(world), ptr(hist), c_int(n), ptr(state), ptr(sel), c_int(rnd),
                               ctypes.byref(active), cur_stream()))
    return active.value


def bkg_grid_nodes(n, grid):
    """Node positions along one axis of n pixels with step `grid` (include/caesar_b200.h, background maps):
    x_i = min(i * grid, n - 1), i = 0 .. ceil((n - 1) / grid)."""
    return [min(i * grid, n - 1) for i in range(-(-(n - 1) // grid) + 1)]


def bkg_grid_init(ncols, R0, R1, row_begin, row_end, box, grid, state, unit_off):
    """cy_bkg_grid_init.  state: uint8 device tensor of >= Nx * Ny cy_noise_state; unit_off: int64 device tensor of
    >= Ny + 1 elements.  Returns the number of work units (synchronises)."""
    units = c_i64(0)
    check(lib.cy_bkg_grid_init(c_int(ncols), c_int(R0), c_int(R1), c_int(row_begin), c_int(row_end), c_int(box),
                               c_int(grid), ptr(state), ptr(unit_off), ctypes.byref(units), cur_stream()))
    return units.value


def bkg_grid_pass(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid, unit_off, units,
                  state, out):
    """cy_bkg_grid_pass: one clipping pass of the grid nodes over this range's rows -> out, uint8 device tensor of
    Nx * Ny cy_noise_partial."""
    check(lib.cy_bkg_grid_pass(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(ncols),
                               c_int(R0), c_int(R1), c_int(row_begin), c_int(row_end), c_int(box), c_int(grid),
                               ptr(unit_off), c_i64(units), ptr(state), ptr(out), cur_stream()))
    return out


def bkg_grid_pass_masked(img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid, unit_off,
                         units, state, out, mask, mask_ncols, mask_col0=0):
    """cy_bkg_grid_pass_masked: bkg_grid_pass with the node-box pixels in the source mask masked; mask: source_mask of
    rows [row_begin, row_end) over mask_ncols columns, region column x = mask column x + mask_col0."""
    check(lib.cy_bkg_grid_pass_masked(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0),
                                      c_int(ncols), c_int(R0), c_int(R1), c_int(row_begin), c_int(row_end), c_int(box),
                                      c_int(grid), ptr(unit_off), c_i64(units), ptr(state), ptr(out), ptr(mask),
                                      c_int(mask_ncols), c_int(mask_col0), cur_stream()))
    return out


def bkg_grid_probe_init(state, nodes, probe):
    """cy_bkg_grid_probe_init: probe state (uint8 device tensor of >= nodes cy_noise_state) with the nodes of nbkg = 0
    active.  Returns their count (synchronises)."""
    n = c_int(0)
    check(lib.cy_bkg_grid_probe_init(ptr(state), c_int(nodes), ptr(probe), ctypes.byref(n), cur_stream()))
    return n.value


def bkg_grid_fill(probe_partials, world, nx, ny, state):
    """cy_bkg_grid_fill: probe partials [world * Nx * Ny * 24] uint8 device (rank-major) -> the holes of the node states
    filled in rings.  Returns the number of nodes filled (synchronises once per ring)."""
    n = c_int(0)
    check(lib.cy_bkg_grid_fill(ptr(probe_partials), c_int(world), c_int(nx), c_int(ny), ptr(state), ctypes.byref(n),
                               cur_stream()))
    return n.value


def bkg_grid_maps(state, ncols, R0, R1, row_begin, row_end, box, grid, bkg, rms):
    """cy_bkg_grid_maps: final node states -> rows [row_begin, row_end) of the bkg and rms maps (device tensors of
    (row_end - row_begin) * ncols 4-byte words, big-endian float32)."""
    check(lib.cy_bkg_grid_maps(ptr(state), c_int(ncols), c_int(R0), c_int(R1), c_int(row_begin), c_int(row_end),
                               c_int(box), c_int(grid), ptr(bkg), ptr(rms), cur_stream()))


def bkg_grid_snr_maps(state, img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box, grid, res,
                      snr):
    """cy_bkg_grid_snr_maps: final node states and this range's image rows (layout as for bkg_grid_pass) -> rows
    [row_begin, row_end) of the background-subtracted and S/N maps (device tensors as for bkg_grid_maps)."""
    check(lib.cy_bkg_grid_snr_maps(ptr(state), ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0),
                                   c_int(ncols), c_int(R0), c_int(R1), c_int(row_begin), c_int(row_end), c_int(box),
                                   c_int(grid), ptr(res), ptr(snr), cur_stream()))


def bkg_grid_sample(state, ncols, R0, R1, box, grid, xy):
    """cy_bkg_grid_sample: final node states (uint8 device tensor) and region pixels xy (int32 device tensor [n, 2] of
    (region column, row)) -> (bkg, rms) float32 device tensors [n], the map values there to the bit (NaN outside)."""
    n = int(xy.shape[0])
    bkg = torch.empty((n,), dtype=torch.float32, device=xy.device)
    rms = torch.empty_like(bkg)
    check(lib.cy_bkg_grid_sample(ptr(state), c_int(ncols), c_int(R0), c_int(R1), c_int(box), c_int(grid), ptr(xy),
                                 c_int(n), ptr(bkg), ptr(rms), cur_stream()))
    return bkg, rms


INJ_DTYPE = np.dtype([('x', '<f8'), ('y', '<f8'), ('peak', '<f8'), ('cx', '<i4'), ('cy', '<i4')])   # cy_injection


def inject_sources(img, row_stride, big_endian, row0, ncols, row_begin, row_end, inj_dev, ninj, rx, ry, icov, saved):
    """cy_inject_sources: the ninj injections inj_dev (uint8 device tensor of INJ_DTYPE records) added to rows
    [row_begin, row_end) of img (layout as for measure_sources); icov = (ixx, ixy, iyy) of C_pix^-1; saved: int32
    device tensor of >= ninj (2 rx + 1)(2 ry + 1) words that receives the original words."""
    check(lib.cy_inject_sources(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(ncols),
                                c_int(row_begin), c_int(row_end), ptr(inj_dev), c_int(ninj), c_int(rx), c_int(ry),
                                c_double(icov[0]), c_double(icov[1]), c_double(icov[2]), ptr(saved), cur_stream()))


def inject_restore(img, row_stride, row0, ncols, row_begin, row_end, inj_dev, ninj, rx, ry, saved):
    """cy_inject_restore: the words inject_sources saved (same arguments) written back."""
    check(lib.cy_inject_restore(ptr(img), c_i64(row_stride), c_int(row0), c_int(ncols), c_int(row_begin),
                                c_int(row_end), ptr(inj_dev), c_int(ninj), c_int(rx), c_int(ry), ptr(saved),
                                cur_stream()))


def negate_rows(img, row_stride, big_endian, row0, ncols, row_begin, row_end):
    """cy_negate_rows: the sign of every finite non-zero pixel of columns [0, ncols) of rows [row_begin, row_end) of img
    (layout as for measure_sources) flipped in place; masked words keep their bits."""
    check(lib.cy_negate_rows(ptr(img), c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(ncols),
                             c_int(row_begin), c_int(row_end), cur_stream()))


def source_peak_snr(state, ncols, R0, R1, box, grid, img, row_stride, big_endian, row0, col_off, src_dev, nsrc, sign,
                    row_begin, row_end, out):
    """cy_source_peak_snr: peak S/N keys of the nsrc sources src_dev (uint8 device tensor of SRC_DTYPE records) over
    rows [row_begin, row_end) of the region of bkg_grid_snr_maps, region column = catalog column - col_off -> out
    (int64 device tensor [nsrc], holding the unsigned keys; decode with peak_snr_decode after an unsigned max fold)."""
    check(lib.cy_source_peak_snr(ptr(state), c_int(ncols), c_int(R0), c_int(R1), c_int(box), c_int(grid), ptr(img),
                                 c_i64(row_stride), c_int(1 if big_endian else 0), c_int(row0), c_int(col_off),
                                 ptr(src_dev), c_int(nsrc), c_int(sign), c_int(row_begin), c_int(row_end), ptr(out),
                                 cur_stream()))
    return out


def peak_snr_decode(keys, ncols, R0, col_off=0):
    """Folded keys of cy_source_peak_snr (uint64 numpy) -> (snr float32, x int64, y int64) in catalog coordinates;
    NaN and -1 where the key is 0 (no pixel)."""
    keys = np.asarray(keys, np.uint64)
    hi = (keys >> np.uint64(32)).astype(np.uint32)
    bits = np.where(hi & np.uint32(0x80000000), hi & np.uint32(0x7fffffff), ~hi).astype(np.uint32)
    idx = (np.uint64(0xffffffff) - (keys & np.uint64(0xffffffff))).astype(np.int64)
    none = keys == 0
    snr = bits.view(np.float32).copy()
    snr[none] = np.nan
    x = np.where(none, -1, idx % ncols + col_off)
    y = np.where(none, -1, idx // ncols + R0)
    return snr, x, y


def to_device_bytes(np_array, device):
    return torch.from_numpy(np_array.view(np.uint8).reshape(-1).copy()).to(device)
