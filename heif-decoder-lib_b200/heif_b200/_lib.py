"""ctypes loader for the in-tree C-ABI library (include/heifcuda.h).

libheifcuda.so (host front-end + sm_100a engine) is required for anything that reconstructs
pixels; libheifcuda_host.so (no CUDA) only offers the parser / container reader and makes every
engine call fail loudly. There is no CPU fallback for the reconstruction path.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)


class Pic(C.Structure):
    """hc_pic (include/heifcuda_records.h)"""
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("crop_x", C.c_int32), ("crop_y", C.c_int32), ("crop_w", C.c_int32), ("crop_h", C.c_int32),
        ("chroma_format", C.c_uint8), ("bit_depth_y", C.c_uint8), ("bit_depth_c", C.c_uint8), ("log2_ctb", C.c_uint8),
        ("ctbs_w", C.c_uint16), ("ctbs_h", C.c_uint16), ("flags", C.c_uint16),
        ("pps_cb_qp_offset", C.c_int8), ("pps_cr_qp_offset", C.c_int8),
        ("colour_primaries", C.c_uint8), ("transfer_characteristics", C.c_uint8), ("matrix_coeffs", C.c_uint8),
        ("full_range", C.c_uint8), ("dst_flags", C.c_uint8), ("pad0", C.c_uint8),
        ("ctu_base", C.c_uint32), ("blk_base", C.c_uint32), ("blk_count", C.c_uint32),
        ("tb_base", C.c_uint32), ("tb_count", C.c_uint32), ("coeff_base", C.c_uint32), ("coeff_count", C.c_uint32),
        ("edge_base", C.c_uint32), ("qp_base", C.c_uint32), ("scaling_base", C.c_uint32),
        ("resid_base", C.c_uint64), ("resid_count", C.c_uint64),
        ("rec_off", C.c_uint64 * 3), ("rec_stride", C.c_uint32 * 3),
        ("dst_off", C.c_uint64 * 3), ("dst_stride", C.c_uint32 * 3),
        ("dst_x", C.c_int32), ("dst_y", C.c_int32), ("dst_w", C.c_int32), ("dst_h", C.c_int32),
    ]


class CscParams(C.Structure):
    """hc_csc_params"""
    _fields_ = [("mode", C.c_int32), ("out_format", C.c_int32), ("full_range", C.c_int32), ("bit_depth", C.c_int32),
                ("r_cr_i", C.c_int32), ("g_cb_i", C.c_int32), ("g_cr_i", C.c_int32), ("b_cb_i", C.c_int32),
                ("r_cr", C.c_float), ("g_cb", C.c_float), ("g_cr", C.c_float), ("b_cb", C.c_float),
                ("in_depth", C.c_int32), ("out_depth", C.c_int32), ("pre_op", C.c_int32), ("post_op", C.c_int32), ("premultiply", C.c_int32), ("upsampling", C.c_int32), ("coeff_matrix", C.c_int32)]


class ImageDesc(C.Structure):
    """hc_image_desc"""
    _fields_ = [(n, C.c_int32) for n in ("width", "height", "chroma_format", "bit_depth", "has_alpha", "out_format",
                                           "bytes_per_pixel", "coded_pictures", "premultiplied_alpha")]


class HeifImageInfo(C.Structure):
    """hc_heif_image_info"""
    _fields_ = [("id", C.c_uint32), ("is_grid", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
                ("rows", C.c_int32), ("cols", C.c_int32), ("alpha_id", C.c_uint32), ("rot", C.c_int32),
                ("mirror", C.c_int32), ("nclx_present", C.c_int32), ("primaries", C.c_int32),
                ("transfer", C.c_int32), ("matrix", C.c_int32), ("full_range", C.c_int32), ("n_transforms", C.c_int32), ("transforms", C.c_uint8 * 8),
                ("has_clap", C.c_int32), ("claps", (C.c_uint32 * 8) * 4), ("premultiplied_alpha", C.c_int32)]


class HeifOverlayInfo(C.Structure):
    """hc_heif_overlay_info"""
    _fields_ = [("canvas_w", C.c_int32), ("canvas_h", C.c_int32), ("background", C.c_uint16 * 4), ("n", C.c_int32),
                ("children", C.c_uint32 * 16), ("dx", C.c_int32 * 16), ("dy", C.c_int32 * 16)]


class StreamStats(C.Structure):
    """hc_stream_stats"""
    _fields_ = [("seconds_total", C.c_double), ("seconds_parse", C.c_double), ("seconds_gpu_phase", C.c_double),
                ("device_ms", C.c_double), ("bytes_h2d", C.c_uint64), ("bytes_d2h", C.c_uint64), ("pixels", C.c_int64),
                ("batches", C.c_int32), ("launches", C.c_int32), ("files_failed", C.c_int32), ("depth", C.c_int32)]


class StreamDest(C.Structure):
    """hc_stream_dest"""
    _fields_ = [("dst", C.c_void_p), ("len", C.c_size_t), ("stride", C.c_size_t)]


IMAGE_CALLBACK = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(ImageDesc), C.c_void_p, C.c_size_t)

# every symbol include/heifcuda.h declares: (name, restype, argtypes)
_vp, _sz, _i, _u32 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint32
SYMBOLS = [
    ("hc_last_error", C.c_char_p, []),
    ("hc_has_cuda_engine", _i, []),
    ("hc_parser_new", _vp, []),
    ("hc_parser_free", None, [_vp]),
    ("hc_parser_push", _i, [_vp, C.c_char_p, _sz, _i]),
    ("hc_parser_take_picture", _vp, [_vp]),
    ("hc_records_free", None, [_vp]),
    ("hc_records_pic", C.POINTER(Pic), [_vp]),
    ("hc_records_ctus", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_blks", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_tbs", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_coeffs", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_edge_map", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_qp_map", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_scaling", _vp, [_vp, C.POINTER(_sz)]),
    ("hc_records_upload_bytes", _sz, [_vp]),
    ("hc_parse_picture", _vp, [C.c_char_p, _sz, _i]),
    ("hc_parse_picture_k0", _vp, [C.c_char_p, _sz, _i]),
    ("hc_k0_prepare", _vp, [C.c_char_p, _sz, _i]),
    ("hc_k0_free", None, [_vp]),
    ("hc_k0_eligible", _i, [_vp]),
    ("hc_k0_why_not", C.c_char_p, [_vp]),
    ("hc_k0_pic", C.POINTER(Pic), [_vp]),
    ("hc_k0_upload_bytes", _sz, [_vp]),
    ("hc_heif_open", _vp, [C.c_char_p, _sz]),
    ("hc_heif_close", None, [_vp]),
    ("hc_heif_primary_id", _u32, [_vp]),
    ("hc_heif_top_level_ids", _i, [_vp, C.POINTER(_u32), _i]),
    ("hc_heif_get_image_info", _i, [_vp, _u32, C.POINTER(HeifImageInfo)]),
    ("hc_heif_get_overlay", _i, [_vp, _u32, C.POINTER(HeifOverlayInfo)]),
    ("hc_heif_grid_tiles", _i, [_vp, _u32, C.POINTER(_u32), _i]),
    ("hc_heif_thumbnail_ids", _i, [_vp, _u32, C.POINTER(_u32), _i]),
    ("hc_heif_auxiliary_ids", _i, [_vp, _u32, _i, C.POINTER(_u32), _i]),
    ("hc_heif_aux_type", _i, [_vp, _u32, C.c_char_p, _sz]),
    ("hc_heif_coded_stream", _i, [_vp, _u32, C.POINTER(_vp), C.POINTER(_sz)]),
    ("hc_free", None, [_vp]),
    ("hc_csc_select", _i, [_i, _i, _i, _i, _i, _i, _i, C.POINTER(CscParams)]),
    ("hc_csc_select_opt", _i, [_i, _i, _i, _i, _i, _i, _i, _i, C.POINTER(CscParams)]),
    ("hc_engine_create", _vp, [_i]),
    ("hc_engine_destroy", None, [_vp]),
    ("hc_engine_set_option", _i, [_vp, C.c_char_p, _i]),
    ("hc_engine_get_option", _i, [_vp, C.c_char_p]),
    ("hc_batch_create", _vp, [_vp]),
    ("hc_batch_destroy", None, [_vp]),
    ("hc_batch_add_canvas", _i, [_vp, _i, _i, _i, _i, _i]),
    ("hc_batch_add_picture", _i, [_vp, _vp, _i, _i, _i, _i, _i]),
    ("hc_batch_add_k0_picture", _i, [_vp, _vp, _i, _i, _i, _i, _i]),
    ("hc_batch_k0_pictures", _i, [_vp]),
    ("hc_batch_set_canvas_transform", _i, [_vp, _i, _i, _i, _i]),
    ("hc_batch_add_canvas_pass", _i, [_vp, _i, _i, _i, _i, _i, _i]),
    ("hc_batch_link_alpha", _i, [_vp, _i, _i]),
    ("hc_batch_set_canvas_output_size", _i, [_vp, _i, _i, _i]),
    ("hc_batch_upload", _i, [_vp]),
    ("hc_batch_reconstruct", _i, [_vp, _i]),
    ("hc_batch_reconstruct_async", _i, [_vp, _i]),
    ("hc_batch_convert", _i, [_vp, _i, C.POINTER(CscParams)]),
    ("hc_batch_convert_many", _i, [_vp, _i, C.POINTER(C.c_int), C.POINTER(CscParams)]),
    ("hc_batch_sync", _i, [_vp]),
    ("hc_batch_read_plane", _i, [_vp, _i, _i, _vp, _sz]),
    ("hc_batch_read_planes", _i, [_vp, _i, _i, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    ("hc_batch_read_rgb", _i, [_vp, _i, _vp, _sz]),
    ("hc_batch_read_rgb_async", _i, [_vp, _i, _vp, _sz]),
    ("hc_batch_copy_rgb_device", _i, [_vp, _i, _vp, _sz]),
    ("hc_batch_read_residual", _i, [_vp, _i, _vp, _sz]),
    ("hc_batch_stage_ms", _i, [_vp, C.POINTER(C.c_float)]),
    ("hc_batch_timer_start", _i, [_vp]),
    ("hc_batch_timer_stop_ms", _i, [_vp, C.POINTER(C.c_float)]),
    ("hc_batch_launch_count", _i, [_vp]),
    ("hc_batch_upload_bytes", _sz, [_vp]),
    ("hc_heic_job_create", _vp, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), _i, _i]),
    ("hc_heic_job_create_items", _vp, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(_u32), _i, _i]),
    ("hc_heic_job_create_band", _vp, [_vp, C.c_char_p, _sz, _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    ("hc_heic_job_copy_rgb_device", _i, [_vp, _i, _vp, _sz]),
    ("hc_heic_job_set_rgb_target", _i, [_vp, _i, _vp, _i]),
    ("hc_batch_set_rgb_target", _i, [_vp, _i, _vp, _sz]),
    ("hc_batch_add_overlay_canvas", _i, [_vp, _i, _i, C.POINTER(C.c_uint16)]),
    ("hc_batch_overlay_add_child", _i, [_vp, _i, _i, _i, _i, C.POINTER(CscParams)]),
    ("hc_shared_image_create", _vp, [_vp, _i, _i, _i]),
    ("hc_shared_image_export", _i, [_vp, C.POINTER(C.c_uint8)]),
    ("hc_shared_image_open", _vp, [_vp, C.POINTER(C.c_uint8), _i, _i, _i]),
    ("hc_shared_image_attach", _vp, [_vp, _vp]),
    ("hc_shared_image_destroy", None, [_vp]),
    ("hc_shared_image_device_ptr", _vp, [_vp]),
    ("hc_shared_image_stride", _sz, [_vp]),
    ("hc_shared_image_read", _i, [_vp, _i, _i, _vp, _sz]),
    ("hc_heic_job_destroy", None, [_vp]),
    ("hc_heic_job_image_count", _i, [_vp]),
    ("hc_heic_job_image_desc", _i, [_vp, _i, C.POINTER(ImageDesc)]),
    ("hc_image_plane_layout", _sz, [C.POINTER(ImageDesc), C.POINTER(_sz), C.POINTER(_sz), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("hc_heic_job_upload", _i, [_vp]),
    ("hc_heic_job_run", _i, [_vp]),
    ("hc_heic_job_sync", _i, [_vp]),
    ("hc_heic_job_read_rgb", _i, [_vp, _i, _vp, _sz]),
    ("hc_heic_job_read_plane", _i, [_vp, _i, _i, _vp, _sz]),
    ("hc_heic_job_stage_ms", _i, [_vp, C.POINTER(C.c_float)]),
    ("hc_heic_job_timer_start", _i, [_vp]),
    ("hc_heic_job_timer_stop_ms", _i, [_vp, C.POINTER(C.c_float)]),
    ("hc_heic_job_launch_count", _i, [_vp]),
    ("hc_heic_job_upload_bytes", _sz, [_vp]),
    ("hc_heic_job_parse_seconds", C.c_double, [_vp]),
    ("hc_heic_decode_stream", _i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), _i, _i, _i, IMAGE_CALLBACK, _vp,
                               C.POINTER(StreamStats)]),
    ("hc_heic_decode_stream_ext", _i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), _i, _i, _i, _vp, C.POINTER(_i), IMAGE_CALLBACK,
                                   _vp, C.POINTER(StreamStats)]),
    ("hc_heic_decode_stream_items", _i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(_u32), _i, _i, _i, _vp, C.POINTER(_i),
                                     IMAGE_CALLBACK, _vp, C.POINTER(StreamStats)]),
    ("hc_host_alloc", _vp, [_sz]),
    ("hc_host_free", None, [_vp]),
]

_libs = {}


def lib_path(host_only=False):
    return os.path.join(_ROOT, "libheifcuda_host.so" if host_only else "libheifcuda.so")


def load(host_only=False):
    """Loads the library. host_only=True loads the CUDA-free build (parser + container only)."""
    if host_only in _libs:
        return _libs[host_only]
    path = lib_path(host_only)
    if not os.path.exists(path):
        raise RuntimeError("%s is missing: run __graft_entry__.build() (make -C heif-decoder-lib_b200/csrc)" % path)
    L = C.CDLL(path)
    for name, res, args in SYMBOLS:
        fn = getattr(L, name)  # AttributeError here means the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _libs[host_only] = L
    return L


class HeifCudaError(RuntimeError):
    pass


def check(L, rc, what):
    if rc is None or (isinstance(rc, int) and rc < 0):
        raise HeifCudaError("%s failed (%s): %s" % (what, rc, (L.hc_last_error() or b"").decode()))
    return rc
