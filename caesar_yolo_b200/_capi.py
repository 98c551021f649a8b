"""ctypes binding of libcaesar_b200.so (include/caesar_b200.h).  No fallback: if the library is missing the
import of any product module fails loudly."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcaesar_b200.so")


class CaesarB200Error(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise CaesarB200Error(
            "libcaesar_b200.so not built (%s). Run `python -m caesar_yolo_b200.build` — there is no CPU fallback."
            % LIB_PATH)
    return ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)


lib = _load()

c_int = ctypes.c_int
c_float = ctypes.c_float
c_double = ctypes.c_double
c_void_p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_uptr = ctypes.c_size_t


class PPConfig(ctypes.Structure):
    """cy_pp_config (include/caesar_b200.h)."""
    _fields_ = [
        ("subtract_bkg", ctypes.c_int32), ("sigma_bkg", c_double), ("use_box_mask_in_bkg", ctypes.c_int32),
        ("bkg_box_mask_fract", c_double), ("bkg_chid", ctypes.c_int32),
        ("clip_shift_data", ctypes.c_int32), ("sigma_clip", c_double), ("clip_chid", ctypes.c_int32),
        ("clip_data", ctypes.c_int32), ("sigma_clip_low", c_double), ("sigma_clip_up", c_double),
        ("nchannels", ctypes.c_int32),
        ("zscale_stretch", ctypes.c_int32), ("zscale_contrasts", c_double * 3),
        ("chan3_preproc", ctypes.c_int32), ("sigma_clip_baseline", c_double),
        ("normalize_minmax", ctypes.c_int32), ("norm_min", c_double), ("norm_max", c_double),
        ("enabled", ctypes.c_int32), ("out_f16", ctypes.c_int32),
    ]


class PPStage(ctypes.Structure):
    """cy_pp_stage."""
    _fields_ = [("type", ctypes.c_int32), ("chid", ctypes.c_int32), ("flag", ctypes.c_int32), ("n", ctypes.c_int32),
                ("p", c_double * 8)]


PP_MAX_STAGES = 16
(PP_BKG_SUB, PP_CLIP_SHIFT, PP_SIGMA_CLIP, PP_CHAN_RESIZE, PP_ZSCALE, PP_CHAN3, PP_MINMAX, PP_ABS_MINMAX, PP_MAX_SCALE,
 PP_ABS_MAX_SCALE, PP_CHAN_MAX_SCALE, PP_MIN_SHIFT, PP_SHIFT, PP_STANDARDIZE, PP_NEG_FIX, PP_LOG_STRETCH, PP_BORDER_MASK,
 PP_HISTEQ) = range(1, 19)


class PPChain(ctypes.Structure):
    """cy_pp_chain: general stage list."""
    _fields_ = [("nstages", ctypes.c_int32), ("out_f16", ctypes.c_int32), ("reject_all", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("st", PPStage * PP_MAX_STAGES)]


class Letterbox(ctypes.Structure):
    """cy_letterbox."""
    _fields_ = [("gain", c_float), ("pad_x", c_float), ("pad_y", c_float), ("w0", ctypes.c_int32),
                ("h0", ctypes.c_int32)]


class RunConfig(ctypes.Structure):
    """cy_run_config (whole-path entry)."""
    _fields_ = [("imgsz", ctypes.c_int32), ("score_thr", c_float), ("iou_thr", c_float), ("thr_soft", c_float),
                ("thr_hard", c_float), ("tile_x", ctypes.c_int32), ("tile_y", ctypes.c_int32), ("step_x", c_double),
                ("step_y", c_double), ("xmin", ctypes.c_int32), ("xmax", ctypes.c_int32), ("ymin", ctypes.c_int32),
                ("ymax", ctypes.c_int32), ("batch_tiles", ctypes.c_int32), ("read_threads", ctypes.c_int32),
                ("rank", ctypes.c_int32), ("world", ctypes.c_int32)]


class SrcPartial(ctypes.Structure):
    """cy_src_partial: one source's sums over one row range."""
    _fields_ = [("npix", c_i64), ("peak_idx", c_i64), ("peak", c_double), ("sum", c_double), ("sw", c_double),
                ("swx", c_double), ("swy", c_double), ("swxx", c_double), ("swyy", c_double), ("swxy", c_double)]


class SrcMeas(ctypes.Structure):
    """cy_src_meas: final per-source measurements."""
    _fields_ = [("npix", c_i64), ("sum", c_double), ("peak", c_double), ("peak_x", c_double), ("peak_y", c_double),
                ("xc", c_double), ("yc", c_double), ("a", c_double), ("b", c_double), ("theta", c_double)]


class NoisePartial(ctypes.Structure):
    """cy_noise_partial: one source's clipped frame sums over one row range and one pass."""
    _fields_ = [("n", c_i64), ("s1", c_double), ("s2", c_double)]


class NoiseState(ctypes.Structure):
    """cy_noise_state: clipping state of one source; bkg, rms, nbkg, iters are final once done."""
    _fields_ = [("lo", c_double), ("hi", c_double), ("c", c_double), ("bkg", c_double), ("rms", c_double),
                ("nbkg", c_i64), ("iters", ctypes.c_int32), ("done", ctypes.c_int32)]


class SelectState(ctypes.Structure):
    """cy_select_state: median select of one source or node (prefixes and ranks of the two middle ranks)."""
    _fields_ = [("prefix", ctypes.c_uint32 * 2), ("rank", c_i64 * 2), ("n", c_i64), ("split", ctypes.c_int32),
                ("round", ctypes.c_int32)]


assert ctypes.sizeof(SrcPartial) == 80 and ctypes.sizeof(SrcMeas) == 80
assert ctypes.sizeof(NoisePartial) == 24 and ctypes.sizeof(NoiseState) == 56 and ctypes.sizeof(SelectState) == 40


ALLGATHER_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                ctypes.c_size_t)


# every exported symbol of include/caesar_b200.h (tests check that the library exports all of them)
SYMBOLS = [
    "cy_last_error", "cy_version", "cy_device_check", "cy_memcpy_d2d", "cy_generate_tiles", "cy_tile_neighbors",
    "cy_letterbox_shape", "cy_preprocess_scratch_bytes", "cy_preprocess", "cy_letterbox_resize", "cy_conv_block_n", "cy_conv2d_nhwc",
    "cy_conv_set_debug", "cy_conv_plan_info", "cy_pp_chain_from_config", "cy_pp_chain_validate",
    "cy_preprocess_chain_scratch_bytes", "cy_preprocess_chain",
    "cy_model_create", "cy_model_set_tensor", "cy_model_set_precision", "cy_model_plan_summary", "cy_letterbox_resize_fmt", "cy_model_finalize", "cy_model_forward", "cy_model_info",
    "cy_stem_conv_nhwc4", "cy_model_profile", "cy_model_conv_bytes", "cy_model_destroy", "cy_num_anchors", "cy_decode_pred", "cy_postprocess_scratch_bytes",
    "cy_postprocess", "cy_nms_scratch_bytes", "cy_nms_batched", "cy_merge_tile", "cy_make_records",
    "cy_compact_scratch_bytes", "cy_compact_records", "cy_merge_global", "cy_measure_sources", "cy_measure_combine",
    "cy_noise_init", "cy_noise_pass", "cy_noise_update", "cy_bkg_grid_init", "cy_bkg_grid_pass", "cy_bkg_grid_maps",
    "cy_bkg_grid_snr_maps", "cy_bkg_grid_sample", "cy_inject_sources", "cy_inject_restore", "cy_negate_rows",
    "cy_source_peak_snr",
    "cy_source_mask", "cy_noise_pass_masked", "cy_bkg_grid_pass_masked", "cy_bkg_grid_probe_init", "cy_bkg_grid_fill",
    "cy_noise_pass_median", "cy_noise_pass_median_masked", "cy_bkg_grid_pass_median", "cy_bkg_grid_pass_median_masked",
    "cy_median_update",
    "cy_ctx_create", "cy_ctx_set_allgather", "cy_ctx_destroy", "cy_run_local", "cy_run_local_payload", "cy_ctx_records",
    "cy_ctx_pack_slot", "cy_ctx_unpack_slots", "cy_run_merge", "cy_run_mosaic", "cy_run_payload", "cy_ctx_info",
]

lib.cy_last_error.restype = ctypes.c_char_p
for _n in ("cy_preprocess_scratch_bytes", "cy_preprocess_chain_scratch_bytes", "cy_postprocess_scratch_bytes", "cy_nms_scratch_bytes",
           "cy_compact_scratch_bytes"):
    getattr(lib, _n).restype = ctypes.c_size_t


def check(rc):
    if rc != 0:
        raise CaesarB200Error("libcaesar_b200 error %d: %s" % (rc, lib.cy_last_error().decode()))
    return rc


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    if t is None:
        return c_void_p(0)
    return c_void_p(t.data_ptr())


def cur_stream():
    import torch
    return c_uptr(torch.cuda.current_stream().cuda_stream)


def cuda_memcpy_d2d(dst, src, nbytes):
    """Device->device copy on torch's current stream (used to read model-owned head buffers in tests)."""
    check(lib.cy_memcpy_d2d(c_void_p(dst), c_void_p(src), ctypes.c_size_t(nbytes), cur_stream()))
