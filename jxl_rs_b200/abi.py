"""ctypes mirror of include/jxg.h (the C ABI of libjxgpu.so).

The structures here are layout-identical to the C header; nothing else in the
package touches raw pointers.
"""
import ctypes as C
import os

JXG_ABI_VERSION = 2

# error codes (include/jxg.h)
JXG_OK = 0
ERRORS = {
    -1: "JXG_ERR_BITSTREAM", -2: "JXG_ERR_UNSUPPORTED", -3: "JXG_ERR_OUT_OF_BOUNDS",
    -4: "JXG_ERR_INVALID_HISTOGRAM_INDEX", -5: "JXG_ERR_INVALID_NUM_NONZEROS",
    -6: "JXG_ERR_RESIDUAL_NONZEROS", -7: "JXG_ERR_ANS_CHECKSUM", -8: "JXG_ERR_INVALID_TRANSFORM",
    -9: "JXG_ERR_INVALID_OUTPUT", -10: "JXG_ERR_LZ77", -20: "JXG_ERR_CUDA", -21: "JXG_ERR_NO_DEVICE",
    -22: "JXG_ERR_ARGUMENT",
}

FORMAT_RGB_U8, FORMAT_RGBA_U8, FORMAT_RGB_F32, FORMAT_XYB_F32_PLANAR, FORMAT_RGB_U16, FORMAT_RGB_F16 = 0, 1, 2, 3, 4, 5
BYTES_PER_PIXEL = {FORMAT_RGB_U8: 3, FORMAT_RGBA_U8: 4, FORMAT_RGB_F32: 12, FORMAT_XYB_F32_PLANAR: 4, FORMAT_RGB_U16: 6,
                   FORMAT_RGB_F16: 6}


class JxgPassDesc(C.Structure):
    _fields_ = [
        ("shift", C.c_uint32), ("use_prefix", C.c_uint32), ("log_alpha_size", C.c_uint32),
        ("num_clusters", C.c_uint32), ("num_contexts", C.c_uint32),
        ("lz77_enabled", C.c_uint32), ("lz77_min_symbol", C.c_uint32), ("lz77_min_length", C.c_uint32),
        ("lz77_length_uint", C.c_uint32), ("lz_dist_cluster", C.c_uint32),
        ("context_map", C.c_void_p), ("uint_configs", C.c_void_p), ("ans_buckets", C.c_void_p),
        ("huff_entries", C.c_void_p), ("huff_offset", C.c_void_p), ("huff_entries_len", C.c_uint32),
        ("coeff_order", C.c_void_p), ("coeff_order_offset", C.c_uint32 * 39), ("coeff_order_len", C.c_uint32),
    ]


class JxgFrameDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32),
        ("global_scale", C.c_uint32), ("x_qm_scale", C.c_uint32), ("b_qm_scale", C.c_uint32),
        ("quant_biases", C.c_float * 4),
        ("base_correlation_x", C.c_float), ("base_correlation_b", C.c_float), ("color_factor", C.c_uint32),
        ("num_qf_thresholds", C.c_uint32), ("qf_thresholds", C.c_uint32 * 15),
        ("num_lf_contexts", C.c_uint32), ("num_block_contexts", C.c_uint32),
        ("block_ctx_map_len", C.c_uint32), ("block_ctx_map", C.c_void_p),
        ("num_histograms", C.c_uint32), ("num_passes", C.c_uint32), ("passes", C.POINTER(JxgPassDesc)),
        ("dequant_tables", C.c_void_p * 17),
        ("lf", C.c_void_p * 3), ("transform_map", C.c_void_p), ("raw_quant_map", C.c_void_p),
        ("epf_map", C.c_void_p), ("quant_lf", C.c_void_p), ("ytox_map", C.c_void_p), ("ytob_map", C.c_void_p),
        ("gab", C.c_uint32), ("gab_w1", C.c_float * 3), ("gab_w2", C.c_float * 3),
        ("epf_iters", C.c_uint32), ("epf_sharp_lut", C.c_float * 8), ("epf_channel_scale", C.c_float * 3),
        ("epf_quant_mul", C.c_float), ("epf_pass0_sigma_scale", C.c_float),
        ("epf_pass2_sigma_scale", C.c_float), ("epf_border_sad_mul", C.c_float),
        ("opsin_inverse_matrix", C.c_float * 9), ("opsin_biases", C.c_float * 3), ("intensity_target", C.c_float),
        ("output_tf", C.c_uint32), ("output_format", C.c_uint32), ("orientation", C.c_uint32),
        ("output_gamma", C.c_float), ("output_luminances", C.c_float * 3),
    ]


class JxgImageInfo(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("num_groups", C.c_uint32),
                ("num_passes", C.c_uint32), ("encoding", C.c_uint32), ("hf_bytes", C.c_uint64),
                ("coded_width", C.c_uint32), ("coded_height", C.c_uint32), ("orientation", C.c_uint32)]


# every symbol include/jxg.h declares (tests check the .so exports all of them)
EXPORTS = [
    "jxg_init", "jxg_shutdown", "jxg_batch_begin", "jxg_batch_add_frame", "jxg_batch_run", "jxg_batch_wait",
    "jxg_batch_rerun_device", "jxg_batch_end", "jxg_batch_read_coeffs", "jxg_batch_read_xyb",
    "jxg_batch_set_debug_stop", "jxg_batch_set_profile", "jxg_batch_stage_times", "jxg_batch_stage_marks", "jxg_batch_stats", "jxg_parse_file", "jxg_parse_file_mt", "jxg_parsed_free", "jxg_parsed_desc",
    "jxg_batch_add_parsed", "jxg_batch_set_deferred_copy", "jxg_last_error", "jxg_device_pci_bus_id",
    "jxg_modular_parse_file", "jxg_modular_parsed_free", "jxg_modular_batch_begin", "jxg_modular_batch_add",
    "jxg_modular_batch_set_lanes", "jxg_modular_batch_run", "jxg_modular_batch_wait", "jxg_modular_batch_rerun_device",
    "jxg_modular_batch_read_planes", "jxg_modular_batch_stats", "jxg_modular_batch_end", "jxg_modular_walk_table",
]

_LIB = None


def library_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libjxgpu.so")


def load_library():
    """Loads libjxgpu.so (built in-tree by __graft_entry__.build()). Fails loudly
    when it is missing: there is no CPU or PyTorch fallback for this path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
                           "the VarDCT hot path has no CPU fallback")
    lib = C.CDLL(path)
    vp, u32p = C.c_void_p, C.POINTER(C.c_uint32)
    lib.jxg_last_error.restype = C.c_char_p
    lib.jxg_init.argtypes = [C.c_int, C.POINTER(vp)]
    lib.jxg_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
    lib.jxg_shutdown.argtypes = [vp]
    lib.jxg_shutdown.restype = None
    lib.jxg_batch_begin.argtypes = [vp, C.c_uint32, C.POINTER(vp)]
    lib.jxg_batch_add_frame.argtypes = [vp, C.POINTER(JxgFrameDesc), vp, vp, vp, C.c_uint32, vp, C.c_size_t, C.c_int]
    lib.jxg_batch_run.argtypes = [vp, vp]
    lib.jxg_batch_wait.argtypes = [vp, u32p, u32p]
    lib.jxg_batch_rerun_device.argtypes = [vp, vp]
    lib.jxg_batch_end.argtypes = [vp]
    lib.jxg_batch_end.restype = None
    lib.jxg_batch_read_coeffs.argtypes = [vp, C.c_uint32, vp, C.c_size_t]
    lib.jxg_batch_read_xyb.argtypes = [vp, C.c_uint32, C.c_int, vp, C.c_size_t]
    lib.jxg_batch_set_debug_stop.argtypes = [vp, C.c_int]
    lib.jxg_batch_set_deferred_copy.argtypes = [vp, C.c_int]
    lib.jxg_modular_parse_file.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(vp), C.POINTER(JxgImageInfo)]
    lib.jxg_modular_parsed_free.argtypes = [vp]
    lib.jxg_modular_parsed_free.restype = None
    lib.jxg_modular_batch_begin.argtypes = [vp, C.POINTER(vp)]
    lib.jxg_modular_batch_add.argtypes = [vp, vp, vp, C.c_size_t, C.c_int]
    lib.jxg_modular_batch_set_lanes.argtypes = [vp, C.c_int]
    lib.jxg_modular_batch_run.argtypes = [vp, vp]
    lib.jxg_modular_batch_wait.argtypes = [vp, u32p, u32p]
    lib.jxg_modular_batch_rerun_device.argtypes = [vp, vp]
    lib.jxg_modular_batch_read_planes.argtypes = [vp, C.c_uint32, vp, C.c_size_t]
    lib.jxg_modular_batch_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                            C.POINTER(C.c_float)]
    lib.jxg_modular_batch_end.argtypes = [vp]
    lib.jxg_modular_walk_table.argtypes = [C.POINTER(C.c_int32), C.c_uint32, C.POINTER(C.c_uint8), C.c_uint32, C.c_uint32,
                                           C.c_uint32, u32p, u32p]
    lib.jxg_modular_batch_end.restype = None
    lib.jxg_batch_set_profile.argtypes = [vp, C.c_int]
    lib.jxg_batch_stage_times.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
    lib.jxg_batch_stage_marks.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
    lib.jxg_batch_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                    C.POINTER(C.c_float)]
    lib.jxg_parse_file.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(vp), C.POINTER(JxgImageInfo)]
    lib.jxg_parse_file_mt.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(vp), C.POINTER(JxgImageInfo)]
    lib.jxg_parsed_free.argtypes = [vp]
    lib.jxg_parsed_free.restype = None
    lib.jxg_parsed_desc.argtypes = [vp, C.c_uint32, C.POINTER(JxgFrameDesc), C.POINTER(vp), C.POINTER(vp),
                                    C.POINTER(vp), u32p]
    lib.jxg_batch_add_parsed.argtypes = [vp, vp, C.c_uint32, vp, C.c_size_t, C.c_int]
    _LIB = lib
    return lib


class JxgError(RuntimeError):
    def __init__(self, code, what=""):
        self.code = code
        super().__init__(f"{ERRORS.get(code, code)}: {what}")


def check(lib, code):
    if code != JXG_OK:
        raise JxgError(code, (lib.jxg_last_error() or b"").decode(errors="replace"))
