"""capi.py -- ctypes binding of libmars_b200.so (the C-ABI boundary).

Mirrors the reference's public interface for the path: the ten mars_* functions of
include/mars_runtime.h:79-138, mars_math.h, the nna_* bring-up calls, plus the additive
mars_b200_* batch entry points (include/mars_b200.h).  No torch types cross this boundary:
buffers are numpy arrays or raw addresses (e.g. `tensor.data_ptr()` of pinned memory).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MARS_B200_LIB") or os.path.join(HERE, "lib", "libmars_b200.so")  # (override: tuning builds, -DMARS_TC_TUNING)


class MarsLibraryMissing(RuntimeError):
    pass


class MarsError(RuntimeError):
    def __init__(self, code, what, detail=""):
        self.code = code
        super().__init__("%s failed: %d (%s)%s" % (what, code, ERR_NAMES.get(code, "?"), (": " + detail) if detail else ""))


ERR_NAMES = {0: "OK", -1: "INVALID_MAGIC", -2: "VERSION_MISMATCH", -3: "ALLOC_FAILED", -4: "INVALID_FILE",
             -5: "NNA_INIT_FAILED", -6: "LAYER_FAILED", -7: "INVALID_TENSOR", -8: "INVALID_LAYER"}


class TensorDesc(C.Structure):
    _pack_ = 1
    _fields_ = [("id", C.c_uint32), ("name", C.c_char * 60), ("dtype", C.c_int32), ("format", C.c_int32),
                ("ndims", C.c_uint32), ("shape", C.c_int32 * 6), ("data_offset", C.c_uint64),
                ("data_size", C.c_uint64), ("scale", C.c_float), ("zero_point", C.c_int32)]


class RuntimeTensor(C.Structure):
    _fields_ = [("desc", TensorDesc), ("vaddr", C.c_void_p), ("paddr", C.c_void_p), ("alloc_size", C.c_size_t),
                ("is_external", C.c_bool)]


class LayerDesc(C.Structure):
    _pack_ = 1
    _fields_ = [("id", C.c_uint32), ("type", C.c_int32), ("num_inputs", C.c_uint32), ("num_outputs", C.c_uint32),
                ("input_tensor_ids", C.c_uint32 * 4), ("output_tensor_ids", C.c_uint32 * 4), ("params", C.c_uint8 * 64)]


class RuntimeLayer(C.Structure):
    _fields_ = [("desc", LayerDesc), ("is_executed", C.c_bool)]


class Header(C.Structure):
    _pack_ = 1
    _fields_ = [("magic", C.c_uint32), ("version_major", C.c_uint16), ("version_minor", C.c_uint16),
                ("flags", C.c_uint32), ("num_layers", C.c_uint32), ("num_tensors", C.c_uint32),
                ("num_inputs", C.c_uint32), ("num_outputs", C.c_uint32), ("weights_offset", C.c_uint64),
                ("weights_size", C.c_uint64), ("input_tensor_ids", C.c_uint32 * 4), ("output_tensor_ids", C.c_uint32 * 4)]


class Model(C.Structure):
    _fields_ = [("header", Header), ("tensors", C.POINTER(RuntimeTensor)), ("layers", C.POINTER(RuntimeLayer)),
                ("ddr_base", C.c_void_p), ("ddr_paddr", C.c_void_p), ("ddr_size", C.c_size_t),
                ("oram_base", C.c_void_p), ("oram_paddr", C.c_void_p), ("oram_size", C.c_size_t),
                ("weights", C.c_void_p), ("weights_size", C.c_size_t), ("total_inference_us", C.c_uint64),
                ("inference_count", C.c_uint32)]


assert C.sizeof(TensorDesc) == 124 and C.sizeof(LayerDesc) == 112 and C.sizeof(Header) == 76

DET_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("w", "<f4"), ("h", "<f4"), ("conf", "<f4"), ("cls", "<i4")])
BOX_DTYPE = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4")])

PM = C.POINTER(Model)


class FRAME(C.Structure):
    """mars_b200_frame_t: one RGB8 frame, rows row_stride bytes apart (0 = w * 3)"""
    _fields_ = [("rgb", C.c_void_p), ("w", C.c_int32), ("h", C.c_int32), ("row_stride", C.c_size_t)]


# colour variants of an NV12 frame (MARS_B200_YUV_*)
YUV_BT601_LIMITED, YUV_BT709_LIMITED, YUV_BT601_FULL, YUV_BT709_FULL = 0, 1, 2, 3


class NV12_FRAME(C.Structure):
    """mars_b200_nv12_frame_t: luma rows y_stride bytes apart (0 = w), ceil(h/2) rows of ceil(w/2) U,V pairs uv_stride bytes
    apart (0 = 2 * ceil(w/2)), colour = YUV_*"""
    _fields_ = [("y", C.c_void_p), ("uv", C.c_void_p), ("w", C.c_int32), ("h", C.c_int32), ("y_stride", C.c_size_t),
                ("uv_stride", C.c_size_t), ("colour", C.c_int32)]


class ROI(C.Structure):
    """mars_b200_roi_t: the w x h pixels at (x, y) of frame `frame` (an index into the call's frame table)"""
    _fields_ = [("frame", C.c_int32), ("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32)]


ROI_DTYPE = np.dtype([("frame", "<i4"), ("x", "<i4"), ("y", "<i4"), ("w", "<i4"), ("h", "<i4")])

# mars_b200_track_box_t: a tracked box of a frame (the filter's box, the matched detection's confidence, class and index)
TRACK_DTYPE = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4"),
                        ("track_id", "<i4"), ("det_index", "<i4")])
MAX_TRACKS = 256  # MARS_B200_MAX_TRACKS


class TRACK_PARAMS(C.Structure):
    """mars_b200_track_params_t; TRACK_PARAMS() holds MARS_B200_TRACK_PARAMS_DEFAULT"""
    _fields_ = [("high_thresh", C.c_float), ("low_thresh", C.c_float), ("new_thresh", C.c_float), ("sim_high", C.c_float),
                ("sim_low", C.c_float), ("sim_unconfirmed", C.c_float), ("max_lost", C.c_int32), ("class_aware", C.c_int32)]
    DEFAULTS = dict(high_thresh=0.5, low_thresh=0.1, new_thresh=0.6, sim_high=0.2, sim_low=0.5, sim_unconfirmed=0.3, max_lost=30,
                    class_aware=0)

    def __init__(self, **kw):
        super().__init__(**{**self.DEFAULTS, **kw})


# zones and counting lines on tracked streams (mars_b200_set_zones)
MAX_ZONES, MAX_ZONE_VERTS, MAX_LINES, MAX_ZONE_EVENTS = 8, 16, 8, 128
ANCHOR_BOTTOM, ANCHOR_CENTRE = 0, 1
ZONE_ENTER, ZONE_DWELL, ZONE_EXIT, ZONE_GONE, CROSS_POS, CROSS_NEG = 0, 1, 2, 3, 4, 5


class ZONE(C.Structure):
    """mars_b200_zone_t: ZONE([(x, y), ...], class_id=-1, anchor=ANCHOR_BOTTOM, min_dwell=0)"""
    _fields_ = [("x", C.c_float * MAX_ZONE_VERTS), ("y", C.c_float * MAX_ZONE_VERTS), ("n_verts", C.c_int32), ("class_id", C.c_int32),
                ("anchor", C.c_int32), ("min_dwell", C.c_int32)]

    def __init__(self, points=(), class_id=-1, anchor=ANCHOR_BOTTOM, min_dwell=0):
        super().__init__(n_verts=len(points), class_id=class_id, anchor=anchor, min_dwell=min_dwell)
        for i, (x, y) in enumerate(points[:MAX_ZONE_VERTS]):
            self.x[i], self.y[i] = x, y


class LINE(C.Structure):
    """mars_b200_line_t: LINE(x0, y0, x1, y1, class_id=-1, anchor=ANCHOR_BOTTOM), directed from (x0, y0) to (x1, y1)"""
    _fields_ = [("x0", C.c_float), ("y0", C.c_float), ("x1", C.c_float), ("y1", C.c_float), ("class_id", C.c_int32), ("anchor", C.c_int32)]

    def __init__(self, x0=0.0, y0=0.0, x1=0.0, y1=0.0, class_id=-1, anchor=ANCHOR_BOTTOM):
        super().__init__(x0, y0, x1, y1, class_id, anchor)


# mars_b200_zone_event_t and mars_b200_zone_frame_t
ZONE_EVENT_DTYPE = np.dtype([("track_id", "<i4"), ("class_id", "<i4"), ("kind", "<i2"), ("index", "<i2"), ("value", "<i4")])
ZONE_FRAME_DTYPE = np.dtype([("frame", "<i4"), ("n_events", "<i4"), ("occupancy", "<i4", MAX_ZONES), ("crossed_pos", "<i4", MAX_LINES),
                             ("crossed_neg", "<i4", MAX_LINES), ("events", ZONE_EVENT_DTYPE, MAX_ZONE_EVENTS)])
assert C.sizeof(ZONE) == 144 and C.sizeof(LINE) == 24 and ZONE_FRAME_DTYPE.itemsize == 2152

# every symbol include/*.h declares: name -> (restype, argtypes)
SIGNATURES = {
    # include/mars_runtime.h
    "mars_load_file": (C.c_int, [C.c_char_p, C.POINTER(PM)]),
    "mars_load_memory": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(PM)]),
    "mars_free": (None, [PM]),
    "mars_get_input": (C.POINTER(RuntimeTensor), [PM, C.c_int]),
    "mars_get_output": (C.POINTER(RuntimeTensor), [PM, C.c_int]),
    "mars_run": (C.c_int, [PM]),
    "mars_get_error_string": (C.c_char_p, [C.c_int]),
    "mars_get_num_inputs": (C.c_int, [PM]),
    "mars_get_num_outputs": (C.c_int, [PM]),
    "mars_print_summary": (None, [PM]),
    # include/mars_math.h
    "mars_vec_add_f32": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "mars_vec_dot_f32": (C.c_float, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "mars_matmul_f32": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t]),
    # include/mxu_ops.h
    "mxu_init": (None, [C.c_void_p]),
    "mxu_is_initialized": (C.c_int, []),
    "mxu_mul_f32": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "mxu_add_f32": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "mxu_sub_f32": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "mxu_relu_f32": (None, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "conv2d_int8_mxu": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                               C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]),
    "conv2d_int8_nhwc_mxu": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]),
    "conv2d_float32_mxu": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    # include/nna.h, include/nna_memory.h
    "nna_init": (C.c_int, []),
    "nna_deinit": (None, []),
    "nna_get_hw_info": (C.c_int, [C.c_void_p]),
    "nna_is_ready": (C.c_int, []),
    "nna_get_version": (C.c_char_p, []),
    "nna_lock": (C.c_int, []),
    "nna_unlock": (C.c_int, []),
    "nna_device_get_ddr": (C.c_void_p, []),
    "nna_device_get_ddr_pbase": (C.c_uint32, []),
    "nna_device_get_oram": (C.c_void_p, []),
    "nna_device_get_fd": (C.c_int, []),
    "nna_device_get_memfd": (C.c_int, []),
    "nna_device_get_nndma_io": (C.c_void_p, []),
    "nna_device_get_nndma_desram": (C.c_void_p, []),
    "nna_malloc": (C.c_void_p, [C.c_size_t]),
    "nna_memalign": (C.c_void_p, [C.c_size_t, C.c_size_t]),
    "nna_calloc": (C.c_void_p, [C.c_size_t, C.c_size_t]),
    "nna_free": (None, [C.c_void_p]),
    "nna_oram_malloc": (C.c_void_p, [C.c_size_t]),
    "nna_oram_free": (None, [C.c_void_p]),
    "nna_oram_get_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nna_cache_flush": (None, [C.c_void_p, C.c_size_t]),
    "nna_cache_invalidate": (None, [C.c_void_p, C.c_size_t]),
    # include/mars_b200.h
    "mars_b200_version": (C.c_char_p, []),
    "mars_b200_device_count": (C.c_int, []),
    "mars_b200_set_device": (C.c_int, [C.c_int]),
    "mars_b200_set_arena_bytes": (None, [C.c_size_t]),
    "mars_b200_last_error": (C.c_char_p, []),
    "mars_b200_arena_upload": (C.c_int, [PM, C.c_int]),
    "mars_b200_arena_download": (C.c_int, [PM, C.c_int, C.c_void_p, C.c_size_t]),
    "mars_b200_arena_clear": (C.c_int, [PM]),
    "mars_b200_run_layer": (C.c_int, [PM, C.c_uint32]),
    "mars_b200_describe": (C.c_size_t, [PM, C.c_char_p, C.c_size_t]),
    "mars_b200_set_opt_level": (None, [PM, C.c_int]),
    "mars_b200_set_depthwise_mode": (None, [PM, C.c_int]),
    "mars_b200_set_strict": (None, [C.c_int]),
    "mars_b200_submit_run_batch": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    "mars_b200_group_load": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "mars_b200_group_free": (None, [C.c_void_p]),
    "mars_b200_group_size": (C.c_int, [C.c_void_p]),
    "mars_b200_group_model": (PM, [C.c_void_p, C.c_int]),
    "mars_b200_group_detect_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_float]),
    "mars_b200_set_f32_mode": (None, [PM, C.c_int]),
    "mars_b200_set_batch": (C.c_int, [PM, C.c_int]),
    "mars_b200_get_batch": (C.c_int, [PM]),
    "mars_b200_input_bytes": (C.c_size_t, [PM]),
    "mars_b200_output_bytes": (C.c_size_t, [PM]),
    "mars_b200_upload_inputs": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "mars_b200_download_outputs": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "mars_b200_preprocess_batch": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int]),
    "mars_b200_run_resident": (C.c_int, [PM, C.c_int, C.c_int]),
    "mars_b200_detect_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_float]),
    "mars_b200_step_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_float, C.c_int]),
    "mars_b200_enqueue_step_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_float, C.c_int]),
    "mars_b200_download_detections": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mars_b200_detect_batch": (C.c_int, [PM, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_float]),
    "mars_b200_submit_batch": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_float]),
    "mars_b200_wait_batch": (C.c_int, [PM, C.c_int]),
    "mars_b200_run_batch": (C.c_int, [PM, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    "mars_b200_detections_device": (None, [PM, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mars_b200_launch_count": (C.c_uint64, [PM]),
    "mars_b200_compute_stream": (C.c_void_p, [PM]),
    "mars_b200_last_gpu_ms": (C.c_float, [PM]),
    "mars_b200_set_profile": (None, [PM, C.c_int]),
    "mars_b200_num_ops": (C.c_int, [PM]),
    "mars_b200_op_info": (C.c_int, [PM, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mars_b200_geometry": (None, [PM, C.c_void_p]),
    "mars_b200_tensor_offset": (C.c_size_t, [PM, C.c_uint32]),
    "mars_yolo_parse_output": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_int]),
    "mars_yolo_nms": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "mars_b200_letterbox": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_letterbox_rgba": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_resize_taps": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mars_b200_plan_describe": (C.c_size_t, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_char_p, C.c_size_t]),
    "mars_b200_requant_fit": (C.c_int, [C.c_float, C.c_longlong, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_longlong)]),
    "mars_b200_requant_ref": (C.c_int, [C.c_int, C.c_float]),
    "mars_b200_requant_variant": (C.c_int, [C.c_float, C.c_longlong]),
    "mars_b200_nmhwsoib2_size": (C.c_size_t, [C.c_int] * 4),
    "mars_b200_ndhwc32_size": (C.c_size_t, [C.c_int] * 4),
    "mars_b200_pack_weights_nmhwsoib2": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_unpack_weights_nmhwsoib2": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_nchw_to_ndhwc32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_ndhwc32_to_nchw": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_pack_weights_nmhwsoib2_device": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mars_b200_unpack_weights_nmhwsoib2_device": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mars_b200_nchw_to_ndhwc32_device": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mars_b200_ndhwc32_to_nchw_device": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mars_yolo_nms_boxes": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "mars_yolo_scale_detections": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "mars_yolo_decode_anchor_grid": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int]),
    "mars_b200_find_yolo_heads": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]),
    "mars_b200_set_yolo_heads": (C.c_int, [PM, C.c_void_p, C.c_int, C.c_float]),
    "mars_b200_find_gfl_heads": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "mars_b200_set_gfl_heads": (C.c_int, [PM, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float]),
    "mars_b200_decode_gfl": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_float, C.c_void_p, C.c_int, C.c_int]),
    "mars_b200_set_frame_size": (C.c_int, [PM, C.c_int, C.c_int, C.c_int, C.c_int]),
    "mars_b200_detect_heads_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_float]),
    "mars_b200_step_heads_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_float]),
    "mars_b200_enqueue_step_heads_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_float]),
    "mars_b200_submit_heads_batch": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_float]),
    "mars_b200_download_boxes": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mars_b200_preprocess_frames": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME)]),
    "mars_b200_preprocess_frames_device": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME)]),
    "mars_b200_submit_frames_heads_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME), C.c_void_p, C.c_void_p, C.c_int,
                                                      C.c_float]),
    "mars_b200_preprocess_frames_nv12": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME)]),
    "mars_b200_preprocess_frames_nv12_device": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME)]),
    "mars_b200_submit_frames_nv12_heads_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME), C.c_void_p, C.c_void_p,
                                                           C.c_int, C.c_float]),
    "mars_b200_yuv_coefficients": (C.c_int, [C.c_int, C.c_void_p]),
    "mars_b200_tile_rois": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "mars_b200_preprocess_rois": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME), C.c_int, C.c_void_p]),
    "mars_b200_preprocess_rois_nv12_device": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME), C.c_int, C.c_void_p]),
    "mars_b200_merge_rois_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_float]),
    "mars_b200_download_frame_boxes": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mars_b200_submit_rois_heads_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                    C.c_int, C.c_float, C.c_float]),
    "mars_b200_submit_rois_nv12_heads_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME), C.c_int, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, C.c_int, C.c_float, C.c_float]),
    "mars_b200_set_tracking": (C.c_int, [PM, C.c_int, C.POINTER(TRACK_PARAMS)]),
    "mars_b200_reset_tracks": (C.c_int, [PM, C.c_int, C.c_int]),
    "mars_b200_track_resident": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_download_tracks": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mars_b200_track_boxes": (C.c_int, [PM, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mars_b200_submit_frames_track_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                      C.c_float]),
    "mars_b200_submit_frames_nv12_track_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME), C.c_void_p, C.c_void_p, C.c_void_p,
                                                           C.c_int, C.c_float]),
    "mars_b200_set_zones": (C.c_int, [PM, C.c_int, C.POINTER(ZONE), C.c_int, C.POINTER(LINE), C.c_int]),
    "mars_b200_download_zones": (C.c_int, [PM, C.c_int, C.c_int, C.c_void_p]),
    "mars_b200_track_boxes_zones": (C.c_int, [PM, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                              C.c_void_p]),
    "mars_b200_submit_frames_zones_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(FRAME), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                      C.c_void_p, C.c_float]),
    "mars_b200_submit_frames_nv12_zones_batch": (C.c_int, [PM, C.c_int, C.c_int, C.POINTER(NV12_FRAME), C.c_void_p, C.c_void_p, C.c_void_p,
                                                           C.c_int, C.c_void_p, C.c_float]),
}

_lib = None


def lib():
    """Load libmars_b200.so and declare every entry point.  Raises if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MarsLibraryMissing(LIB_PATH + " is missing: run `make -C thingino-accel_b200/csrc` "
                                     "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)  # AttributeError = header/library drift
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def _addr(buf):
    """numpy array / int address / object with data_ptr() -> raw address"""
    if buf is None:
        return None
    if isinstance(buf, int):
        return buf
    if isinstance(buf, np.ndarray):
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):
        return buf.data_ptr()
    raise TypeError(type(buf))


def host_frames(frames):
    """[h, w, 3] uint8 arrays -> (FRAME table, the arrays it points into).  A view whose rows are further apart than w * 3
    (strides (pitch, 3, 1), e.g. a crop of a wider buffer) passes its pitch; any other layout is copied first."""
    table = (FRAME * len(frames))()
    keep = []
    for i, f in enumerate(frames):
        a = np.asarray(f)
        h, w, c = a.shape
        assert c == 3 and a.dtype == np.uint8
        if not (a.strides[1:] == (3, 1) and a.strides[0] >= 3 * w):
            a = np.ascontiguousarray(a)
        keep.append(a)
        table[i] = FRAME(a.ctypes.data, w, h, a.strides[0])
    return table, keep


def device_frames(frames):
    """[(ptr, w, h, row_stride), ...] of frames in device memory -> FRAME table"""
    table = (FRAME * len(frames))()
    for i, (p, w, h, stride) in enumerate(frames):
        table[i] = FRAME(p, w, h, stride)
    return table


def host_nv12_frames(frames):
    """[(y, uv, colour), ...] with y a [h, w] uint8 array and uv a [ceil(h/2), ceil(w/2), 2] uint8 array -> (NV12_FRAME table,
    the arrays it points into).  Views whose rows are further apart than their width (strides (pitch, 1) and (pitch, 2, 1))
    pass their pitches; any other layout is copied first."""
    table = (NV12_FRAME * len(frames))()
    keep = []
    for i, (y, uv, colour) in enumerate(frames):
        y, uv = np.asarray(y), np.asarray(uv)
        h, w = y.shape
        assert y.dtype == np.uint8 and uv.dtype == np.uint8 and uv.shape == ((h + 1) // 2, (w + 1) // 2, 2), (y.shape, uv.shape)
        if not (y.strides[1] == 1 and y.strides[0] >= w):
            y = np.ascontiguousarray(y)
        if not (uv.strides[1:] == (2, 1) and uv.strides[0] >= uv.shape[1] * 2):
            uv = np.ascontiguousarray(uv)
        keep += [y, uv]
        table[i] = NV12_FRAME(y.ctypes.data, uv.ctypes.data, w, h, y.strides[0], uv.strides[0], colour)
    return table, keep


def device_nv12_frames(frames):
    """[(y_ptr, uv_ptr, w, h, y_stride, uv_stride, colour), ...] of NV12 frames in device memory -> NV12_FRAME table"""
    table = (NV12_FRAME * len(frames))()
    for i, f in enumerate(frames):
        table[i] = NV12_FRAME(*f)
    return table


def roi_table(rois):
    """[(frame, x, y, w, h), ...] or a ROI_DTYPE array -> contiguous ROI_DTYPE array (the layout of mars_b200_roi_t)"""
    if isinstance(rois, np.ndarray) and rois.dtype == ROI_DTYPE:
        return np.ascontiguousarray(rois)
    return np.array([tuple(int(v) for v in r) for r in rois], dtype=ROI_DTYPE)


def _numel(desc):
    n = 1
    for i in range(min(desc.ndims, 6)):
        n *= max(desc.shape[i], 0)
    return n


class MarsModel:
    """A loaded .mars model (mars_load_memory ... mars_free), plus the batch entry points."""

    def __init__(self, model, arena_bytes=0, device=None, batch=1):
        L = lib()
        if device is not None:
            if L.mars_b200_set_device(device) != 0:
                raise MarsError(-5, "mars_b200_set_device", L.mars_b200_last_error().decode())
        L.mars_b200_set_arena_bytes(arena_bytes)
        self.m = PM()
        self._inflight = {}  # pool -> what a submitted batch reads until wait_batch
        if isinstance(model, (bytes, bytearray, memoryview)):
            self._blob = bytes(model)
            err = L.mars_load_memory(self._blob, len(self._blob), C.byref(self.m))
        else:
            err = L.mars_load_file(os.fsencode(model), C.byref(self.m))
        L.mars_b200_set_arena_bytes(0)
        if err != 0:
            raise MarsError(err, "mars_load", L.mars_b200_last_error().decode())
        g = (C.c_size_t * 5)()
        L.mars_b200_geometry(self.m, g)
        self.weights_size, self.buffer_size, self.num_buffers, self.slot_stride, self.arena_bytes = [int(v) for v in g]
        if batch != 1:
            self.set_batch(batch)

    # ---- reference-shaped accessors ------------------------------------------------
    @property
    def header(self):
        return self.m.contents.header

    def _check(self, err, what):
        if err != 0:
            raise MarsError(err, what, lib().mars_b200_last_error().decode())

    def input(self, i=0):
        p = lib().mars_get_input(self.m, i)
        return p.contents if p else None

    def output(self, i=0):
        p = lib().mars_get_output(self.m, i)
        return p.contents if p else None

    def tensor_view(self, rt, nbytes=None):
        n = rt.alloc_size if nbytes is None else nbytes
        return np.ctypeslib.as_array((C.c_uint8 * n).from_address(rt.vaddr))

    def set_input(self, data, i=0):
        t = self.input(i)
        raw = np.ascontiguousarray(data).view(np.uint8).ravel()
        assert raw.size <= t.alloc_size
        self.tensor_view(t)[: raw.size] = raw

    def output_bytes(self, i=0):
        o = self.output(i)
        es = {0: 4, 1: 4, 2: 2}.get(o.desc.dtype, 1)
        return self.tensor_view(o, _numel(o.desc) * es)

    def run(self):
        self._check(lib().mars_run(self.m), "mars_run")

    def mirror(self):
        """host mirror of the whole arena (ddr_base)"""
        return np.ctypeslib.as_array((C.c_uint8 * self.arena_bytes).from_address(self.m.contents.ddr_base))

    def tensor_offset(self, idx):
        return int(lib().mars_b200_tensor_offset(self.m, idx))

    # ---- B200 additions ------------------------------------------------------------
    def set_batch(self, n):
        self._check(lib().mars_b200_set_batch(self.m, n), "mars_b200_set_batch")

    def set_opt_level(self, lvl):
        lib().mars_b200_set_opt_level(self.m, lvl)

    def set_f32_mode(self, mode):
        lib().mars_b200_set_f32_mode(self.m, mode)

    def set_depthwise_mode(self, mode):
        lib().mars_b200_set_depthwise_mode(self.m, mode)

    def arena_upload(self, slot=0):
        self._check(lib().mars_b200_arena_upload(self.m, slot), "arena_upload")

    def arena_download(self, slot=0):
        n = min(self.arena_bytes, self.weights_size + self.num_buffers * self.buffer_size)
        out = np.zeros(n, dtype=np.uint8)
        self._check(lib().mars_b200_arena_download(self.m, slot, out.ctypes.data, n), "arena_download")
        return out

    def arena_clear(self):
        self._check(lib().mars_b200_arena_clear(self.m), "arena_clear")

    def run_layer(self, i):
        return lib().mars_b200_run_layer(self.m, i)

    def describe(self):
        n = lib().mars_b200_describe(self.m, None, 0)
        buf = C.create_string_buffer(n + 1)
        lib().mars_b200_describe(self.m, buf, n + 1)
        return buf.value.decode()

    @property
    def input_bytes(self):
        return int(lib().mars_b200_input_bytes(self.m))

    @property
    def out_bytes(self):
        return int(lib().mars_b200_output_bytes(self.m))

    def upload_inputs(self, first, n, host, stride=0):
        self._check(lib().mars_b200_upload_inputs(self.m, first, n, _addr(host), stride), "upload_inputs")

    def preprocess(self, first, frames):
        """frames: [n, h, w, 3] uint8 (host) -> letterboxed into input tensor 0 of slots [first, first+n) on the device
        (reference src/mars/mars_yolo_test.c:40-77); returns the GPU milliseconds of the copy + kernels"""
        f = np.ascontiguousarray(frames, dtype=np.uint8)
        n, h, w, c = f.shape
        assert c == 3
        self._check(lib().mars_b200_preprocess_batch(self.m, first, n, f.ctypes.data, h * w * 3, w, h), "preprocess_batch")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def preprocess_frames(self, first, frames):
        """frames: list of [h, w, 3] uint8 host arrays of any sizes -> letterboxed into input tensor 0 of slots
        [first, first+len(frames)) in one pass; returns the GPU milliseconds of the copies + kernels"""
        table, _keep = host_frames(frames)
        self._check(lib().mars_b200_preprocess_frames(self.m, first, len(frames), table), "preprocess_frames")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def preprocess_frames_device(self, first, frames):
        """frames: [(device ptr, w, h, row_stride), ...]; enqueued on compute_stream(), which the caller synchronises with"""
        self._check(lib().mars_b200_preprocess_frames_device(self.m, first, len(frames), device_frames(frames)),
                    "preprocess_frames_device")

    def preprocess_frames_nv12(self, first, frames):
        """frames: list of (y, uv, colour) NV12 host frames of any sizes (host_nv12_frames) -> letterboxed into input tensor 0 of
        slots [first, first+len(frames)) in one pass; returns the GPU milliseconds of the copies + kernels"""
        table, _keep = host_nv12_frames(frames)
        self._check(lib().mars_b200_preprocess_frames_nv12(self.m, first, len(frames), table), "preprocess_frames_nv12")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def preprocess_frames_nv12_device(self, first, frames):
        """frames: [(y_ptr, uv_ptr, w, h, y_stride, uv_stride, colour), ...] in device memory; enqueued on compute_stream()"""
        self._check(lib().mars_b200_preprocess_frames_nv12_device(self.m, first, len(frames), device_nv12_frames(frames)),
                    "preprocess_frames_nv12_device")

    # ---- tiled detection: regions of frames, merged per frame (include/mars_b200.h) -------------
    def preprocess_rois(self, first, frames, rois):
        """frames: list of [h, w, 3] uint8 host arrays (row-strided views pass their pitch); rois: (frame, x, y, w, h) per region
        (tile_rois) -> region r letterboxed into slot first + r; returns the GPU milliseconds of the copies + kernels"""
        table, _keep = host_frames(frames)
        r = roi_table(rois)
        self._check(lib().mars_b200_preprocess_rois(self.m, first, len(frames), table, len(r), r.ctypes.data), "preprocess_rois")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def preprocess_rois_nv12_device(self, first, frames, rois):
        """frames: [(y_ptr, uv_ptr, w, h, y_stride, uv_stride, colour), ...] in device memory; enqueued on compute_stream()"""
        r = roi_table(rois)
        self._check(lib().mars_b200_preprocess_rois_nv12_device(self.m, first, len(frames), device_nv12_frames(frames), len(r), r.ctypes.data),
                    "preprocess_rois_nv12_device")

    def merge_rois_resident(self, first, n_frames, rois, merge_thresh=0.45):
        """after a heads step on slots [first, first + len(rois)): boxes of each frame's regions shifted into the frame and merged
        by the corner NMS into frame records [first, first + n_frames); enqueued on compute_stream()"""
        r = roi_table(rois)
        self._check(lib().mars_b200_merge_rois_resident(self.m, first, n_frames, len(r), r.ctypes.data, merge_thresh), "merge_rois_resident")

    def download_frame_boxes(self, first, n, maxd=1000):
        boxes = np.zeros((n, maxd), dtype=BOX_DTYPE)
        counts = np.zeros(n, dtype=np.int32)
        self._check(lib().mars_b200_download_frame_boxes(self.m, first, n, boxes.ctypes.data, counts.ctypes.data, maxd), "download_frame_boxes")
        return boxes, counts

    def submit_rois_heads_batch(self, pool, frames, rois, boxes, counts, maxd=1000, thresh=0.45, merge_thresh=0.45):
        """the tiled flow on one pool from [h, w, 3] uint8 host frames: boxes [len(frames), maxd] in frame coordinates.  The frames
        and regions are kept alive until wait_batch(pool); boxes and counts must be kept alive by the caller"""
        table, keep = host_frames(frames)
        r = roi_table(rois)
        self._check(lib().mars_b200_submit_rois_heads_batch(self.m, pool, len(frames), table, len(r), r.ctypes.data, _addr(boxes), _addr(counts),
                                                            maxd, thresh, merge_thresh), "submit_rois_heads_batch")
        self._inflight[pool] = (table, keep, r)

    def submit_rois_nv12_heads_batch(self, pool, frames, rois, boxes, counts, maxd=1000, thresh=0.45, merge_thresh=0.45):
        """submit_rois_heads_batch from (y, uv, colour) NV12 host frames (host_nv12_frames)"""
        table, keep = host_nv12_frames(frames)
        r = roi_table(rois)
        self._check(lib().mars_b200_submit_rois_nv12_heads_batch(self.m, pool, len(frames), table, len(r), r.ctypes.data, _addr(boxes),
                                                                 _addr(counts), maxd, thresh, merge_thresh), "submit_rois_nv12_heads_batch")
        self._inflight[pool] = (table, keep, r)

    # ---- multi-object tracking of camera streams (include/mars_b200.h) --------------------------------
    def set_tracking(self, n_streams, params=None, **kw):
        """tracker state for n_streams streams, all reset; params: TRACK_PARAMS, or its fields as keywords (the rest default);
        n_streams = 0 frees it"""
        p = params if params is not None else TRACK_PARAMS(**kw)
        self._check(lib().mars_b200_set_tracking(self.m, n_streams, C.byref(p)), "set_tracking")

    def reset_tracks(self, first_stream, n):
        """streams [first_stream, first_stream + n) start over; enqueued on compute_stream()"""
        self._check(lib().mars_b200_reset_tracks(self.m, first_stream, n), "reset_tracks")

    def track_resident(self, first, streams):
        """after a heads step on slots [first, first + len(streams)): slot first + i is the next frame of stream streams[i];
        enqueued on compute_stream()"""
        s = np.ascontiguousarray(streams, dtype=np.int32)
        self._check(lib().mars_b200_track_resident(self.m, first, s.size, s.ctypes.data), "track_resident")

    def download_tracks(self, first, n, maxd=MAX_TRACKS):
        out = np.zeros((n, maxd), dtype=TRACK_DTYPE)
        counts = np.zeros(n, dtype=np.int32)
        self._check(lib().mars_b200_download_tracks(self.m, first, n, out.ctypes.data, counts.ctypes.data, maxd), "download_tracks")
        return out, counts

    def track_boxes(self, streams, boxes, maxd=MAX_TRACKS):
        """boxes: one BOX_DTYPE array per entry, the next frame of stream streams[i] -> (TRACK_DTYPE [n, maxd], counts [n]);
        synchronous"""
        return self._track_boxes(streams, boxes, maxd, False)

    def track_boxes_zones(self, streams, boxes, maxd=MAX_TRACKS):
        """track_boxes plus the zone record of every entry -> (TRACK_DTYPE [n, maxd], counts [n], ZONE_FRAME_DTYPE [n])"""
        return self._track_boxes(streams, boxes, maxd, True)

    def _track_boxes(self, streams, boxes, maxd, zones):
        s = np.ascontiguousarray(streams, dtype=np.int32)
        n = s.size
        counts = np.array([len(b) for b in boxes], dtype=np.int32)
        stride = max(1, int(counts.max()) if n else 1)
        table = np.zeros((n, stride), dtype=BOX_DTYPE)
        for i, b in enumerate(boxes):
            table[i, : len(b)] = b
        out = np.zeros((n, maxd), dtype=TRACK_DTYPE)
        oc = np.zeros(n, dtype=np.int32)
        zo = np.zeros(n, dtype=ZONE_FRAME_DTYPE) if zones else None
        self._check(lib().mars_b200_track_boxes_zones(self.m, n, s.ctypes.data, table.ctypes.data, counts.ctypes.data, stride, out.ctypes.data,
                                                      oc.ctypes.data, maxd, None if zo is None else zo.ctypes.data), "track_boxes")
        return (out, oc, zo) if zones else (out, oc)

    def set_zones(self, stream, zones=(), lines=()):
        """geometry of tracker stream `stream` (ZONE and LINE sequences); its analytics start over; empty: the stream is off"""
        za, la = (ZONE * max(1, len(zones)))(*zones), (LINE * max(1, len(lines)))(*lines)
        self._check(lib().mars_b200_set_zones(self.m, stream, za, len(zones), la, len(lines)), "set_zones")

    def download_zones(self, first, n):
        """zone records of track records [first, first + n) -> ZONE_FRAME_DTYPE [n]"""
        out = np.zeros(n, dtype=ZONE_FRAME_DTYPE)
        self._check(lib().mars_b200_download_zones(self.m, first, n, out.ctypes.data), "download_zones")
        return out

    def submit_frames_track_batch(self, pool, frames, streams, out, counts, maxd=MAX_TRACKS, thresh=0.45):
        """submit_frames_heads_batch followed by the tracker: frame i is the next frame of stream streams[i]; out [n, maxd] TRACK_DTYPE.
        The frames and the stream table are kept alive until wait_batch(pool); out and counts must be kept alive by the caller"""
        table, keep = host_frames(frames)
        s = np.ascontiguousarray(streams, dtype=np.int32)
        self._check(lib().mars_b200_submit_frames_track_batch(self.m, pool, len(frames), table, s.ctypes.data, _addr(out), _addr(counts), maxd,
                                                              thresh), "submit_frames_track_batch")
        self._inflight[pool] = (table, keep, s)

    def submit_frames_nv12_track_batch(self, pool, frames, streams, out, counts, maxd=MAX_TRACKS, thresh=0.45):
        """submit_frames_track_batch from (y, uv, colour) NV12 host frames (host_nv12_frames)"""
        table, keep = host_nv12_frames(frames)
        s = np.ascontiguousarray(streams, dtype=np.int32)
        self._check(lib().mars_b200_submit_frames_nv12_track_batch(self.m, pool, len(frames), table, s.ctypes.data, _addr(out), _addr(counts),
                                                                   maxd, thresh), "submit_frames_nv12_track_batch")
        self._inflight[pool] = (table, keep, s)

    def submit_frames_zones_batch(self, pool, frames, streams, out, counts, zones, maxd=MAX_TRACKS, thresh=0.45):
        """submit_frames_track_batch plus the zone record of every frame into zones [n] ZONE_FRAME_DTYPE, read back in the same
        batch; out, counts and zones must be kept alive by the caller until wait_batch(pool)"""
        table, keep = host_frames(frames)
        s = np.ascontiguousarray(streams, dtype=np.int32)
        self._check(lib().mars_b200_submit_frames_zones_batch(self.m, pool, len(frames), table, s.ctypes.data, _addr(out), _addr(counts), maxd,
                                                              _addr(zones), thresh), "submit_frames_zones_batch")
        self._inflight[pool] = (table, keep, s)

    def submit_frames_nv12_zones_batch(self, pool, frames, streams, out, counts, zones, maxd=MAX_TRACKS, thresh=0.45):
        """submit_frames_zones_batch from (y, uv, colour) NV12 host frames (host_nv12_frames)"""
        table, keep = host_nv12_frames(frames)
        s = np.ascontiguousarray(streams, dtype=np.int32)
        self._check(lib().mars_b200_submit_frames_nv12_zones_batch(self.m, pool, len(frames), table, s.ctypes.data, _addr(out), _addr(counts),
                                                                   maxd, _addr(zones), thresh), "submit_frames_nv12_zones_batch")
        self._inflight[pool] = (table, keep, s)

    def download_outputs(self, first, n, host=None, stride=0):
        if host is None:
            host = np.zeros((n, self.out_bytes), dtype=np.uint8)
        self._check(lib().mars_b200_download_outputs(self.m, first, n, _addr(host), stride), "download_outputs")
        return host

    def run_resident(self, first, n):
        self._check(lib().mars_b200_run_resident(self.m, first, n), "run_resident")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def detect_resident(self, first, n, thresh=0.45):
        self._check(lib().mars_b200_detect_resident(self.m, first, n, thresh), "detect_resident")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def step_resident(self, first, n, thresh=0.45, with_detect=True):
        self._check(lib().mars_b200_step_resident(self.m, first, n, thresh, 1 if with_detect else 0), "step_resident")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def enqueue_step_resident(self, first, n, thresh=0.45, with_detect=True):
        """step_resident without the host synchronisation: the work is on compute_stream() when this returns"""
        self._check(lib().mars_b200_enqueue_step_resident(self.m, first, n, thresh, 1 if with_detect else 0), "enqueue_step_resident")

    def compute_stream(self):
        """cudaStream_t handle (int) of the stream the model's kernels run on"""
        return int(lib().mars_b200_compute_stream(self.m) or 0)

    def download_detections(self, first, n, maxd=1000):
        dets = np.zeros((n, maxd), dtype=DET_DTYPE)
        counts = np.zeros(n, dtype=np.int32)
        self._check(lib().mars_b200_download_detections(self.m, first, n, dets.ctypes.data, counts.ctypes.data, maxd),
                    "download_detections")
        return dets, counts

    def detect_batch(self, n, inputs, in_stride, dets, counts, maxd=1000, thresh=0.45):
        self._check(lib().mars_b200_detect_batch(self.m, n, _addr(inputs), in_stride, _addr(dets), _addr(counts), maxd, thresh),
                    "detect_batch")

    def submit_batch(self, pool, n, inputs, in_stride, dets, counts, maxd=1000, thresh=0.45):
        """queue a batch on half `pool` of the slot pool; buffers must stay alive until wait_batch(pool)"""
        self._check(lib().mars_b200_submit_batch(self.m, pool, n, _addr(inputs), in_stride, _addr(dets), _addr(counts), maxd, thresh),
                    "submit_batch")

    def submit_run_batch(self, pool, n, inputs, in_stride, outputs, out_stride):
        """queue a batch without the YOLO post-process (raw output tensors read back); wait with wait_batch(pool)"""
        self._check(lib().mars_b200_submit_run_batch(self.m, pool, n, _addr(inputs), in_stride, _addr(outputs), out_stride), "submit_run_batch")

    # ---- YOLOv5 Detect heads (include/mars_b200.h) ------------------------------------
    def set_yolo_heads(self, tensor_ids=None, conf_thresh=0.25, enable=True):
        """decode the three head convs inside every run (tensor_ids None: find them); enable=False switches it off"""
        if not enable:
            ids, n = None, 0
        elif tensor_ids is None:
            ids, n = None, 3
        else:
            ids = np.ascontiguousarray(tensor_ids, dtype=np.uint32)
            n = ids.size
        self._check(lib().mars_b200_set_yolo_heads(self.m, None if ids is None else ids.ctypes.data, n, conf_thresh), "set_yolo_heads")

    def set_gfl_heads(self, tensor_ids=None, nc=80, reg_max=7, centre="half", conf_thresh=0.25, enable=True):
        """decode NanoDet GFL head convs (3 or 4 levels, nc + 4 (reg_max + 1) channels) inside every run, replacing YOLO heads if set;
        tensor_ids None: find them; centre "half" (NanoDet-m) or "corner" (NanoDet-Plus); enable=False switches decoding off"""
        if not enable:
            ids, n = None, 0
        elif tensor_ids is None:
            ids, n = None, 3
        else:
            ids = np.ascontiguousarray(tensor_ids, dtype=np.uint32)
            n = ids.size
        code = GFL_CENTRE[centre] if isinstance(centre, str) else int(centre)
        self._check(lib().mars_b200_set_gfl_heads(self.m, None if ids is None else ids.ctypes.data, n, nc, reg_max, code, conf_thresh),
                    "set_gfl_heads")

    def set_frame_size(self, first, n, w, h):
        """original frame size of slots [first, first+n) for the letterbox inverse (0, 0: network coordinates)"""
        self._check(lib().mars_b200_set_frame_size(self.m, first, n, w, h), "set_frame_size")

    def detect_heads_resident(self, first, n, thresh=0.45):
        self._check(lib().mars_b200_detect_heads_resident(self.m, first, n, thresh), "detect_heads_resident")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def step_heads_resident(self, first, n, thresh=0.45):
        self._check(lib().mars_b200_step_heads_resident(self.m, first, n, thresh), "step_heads_resident")
        return float(lib().mars_b200_last_gpu_ms(self.m))

    def enqueue_step_heads_resident(self, first, n, thresh=0.45):
        self._check(lib().mars_b200_enqueue_step_heads_resident(self.m, first, n, thresh), "enqueue_step_heads_resident")

    def submit_heads_batch(self, pool, n, inputs, in_stride, boxes, counts, maxd=1000, thresh=0.45):
        """submit_batch with the heads decode: boxes [n, maxd] BOX_DTYPE; buffers must stay alive until wait_batch(pool)"""
        self._check(lib().mars_b200_submit_heads_batch(self.m, pool, n, _addr(inputs), in_stride, _addr(boxes), _addr(counts), maxd, thresh),
                    "submit_heads_batch")

    def submit_frames_heads_batch(self, pool, frames, boxes, counts, maxd=1000, thresh=0.45):
        """submit_heads_batch from a list of [h, w, 3] uint8 host frames of any sizes; boxes in frame coordinates.  The
        frames are kept alive until wait_batch(pool); boxes and counts must be kept alive by the caller"""
        table, keep = host_frames(frames)
        self._check(lib().mars_b200_submit_frames_heads_batch(self.m, pool, len(frames), table, _addr(boxes), _addr(counts), maxd, thresh),
                    "submit_frames_heads_batch")
        self._inflight[pool] = (table, keep)

    def submit_frames_nv12_heads_batch(self, pool, frames, boxes, counts, maxd=1000, thresh=0.45):
        """submit_frames_heads_batch from a list of (y, uv, colour) NV12 host frames (host_nv12_frames).  The frames are kept
        alive until wait_batch(pool); boxes and counts must be kept alive by the caller"""
        table, keep = host_nv12_frames(frames)
        self._check(lib().mars_b200_submit_frames_nv12_heads_batch(self.m, pool, len(frames), table, _addr(boxes), _addr(counts), maxd,
                                                                   thresh), "submit_frames_nv12_heads_batch")
        self._inflight[pool] = (table, keep)

    def download_boxes(self, first, n, maxd=1000):
        boxes = np.zeros((n, maxd), dtype=BOX_DTYPE)
        counts = np.zeros(n, dtype=np.int32)
        self._check(lib().mars_b200_download_boxes(self.m, first, n, boxes.ctypes.data, counts.ctypes.data, maxd), "download_boxes")
        return boxes, counts

    def wait_batch(self, pool):
        try:
            self._check(lib().mars_b200_wait_batch(self.m, pool), "wait_batch")
        finally:
            self._inflight.pop(pool, None)

    def run_batch(self, n, inputs, in_stride, outputs, out_stride):
        self._check(lib().mars_b200_run_batch(self.m, n, _addr(inputs), in_stride, _addr(outputs), out_stride), "run_batch")

    def detections_device(self):
        """(dets_ptr, counts_ptr, stride) of the device-resident detection records"""
        d, c, s = C.c_void_p(), C.c_void_p(), C.c_int()
        lib().mars_b200_detections_device(self.m, C.byref(d), C.byref(c), C.byref(s))
        return d.value, c.value, s.value

    @property
    def last_gpu_ms(self):
        return float(lib().mars_b200_last_gpu_ms(self.m))

    @property
    def launch_count(self):
        return int(lib().mars_b200_launch_count(self.m))

    def set_profile(self, on):
        lib().mars_b200_set_profile(self.m, 1 if on else 0)

    def op_profile(self):
        """list of dicts, one per device op, with accumulated CUDA-event milliseconds"""
        out = []
        info = (C.c_int32 * 16)()
        ms, calls, n = C.c_double(), C.c_uint64(), C.c_uint64()
        for i in range(lib().mars_b200_num_ops(self.m)):
            lib().mars_b200_op_info(self.m, i, info, C.byref(ms), C.byref(calls), C.byref(n))
            out.append(dict(op=i, kind=info[0], layer=info[1], impl=info[2], mode=info[3], ic=info[4], oc=info[5], oh=info[6],
                            ow=info[7], kh=info[8], kw=info[9], fused=info[10], ih=info[11], iw=info[12], ms=ms.value,
                            calls=calls.value, n=n.value))
        return out

    def close(self):
        if self.m:
            lib().mars_free(self.m)
            self.m = PM()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- pre-process on host arrays ------------------------------------------------------
def letterbox(rgb, tw, th, nhwc=False):
    """[h, w, 3] uint8 frame -> tw*th*3 int8 network input (runs on the device; reference load_image minus the decode)"""
    f = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = f.shape
    out = np.zeros(tw * th * 3, dtype=np.int8)
    if lib().mars_b200_letterbox(f.ctypes.data, w, h, tw, th, 1 if nhwc else 0, out.ctypes.data) != 0:
        raise RuntimeError("mars_b200_letterbox failed: " + lib().mars_b200_last_error().decode())
    return out


def letterbox_rgba(rgb, tw=640, th=640):
    """[h, w, 3] uint8 frame -> tw*th*4 uint8 RGBA frame (reference examples/yolo_detect.cpp:72-130 minus the decode)"""
    f = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = f.shape
    out = np.zeros(tw * th * 4, dtype=np.uint8)
    if lib().mars_b200_letterbox_rgba(f.ctypes.data, w, h, tw, th, out.ctypes.data) != 0:
        raise RuntimeError("mars_b200_letterbox_rgba failed: " + lib().mars_b200_last_error().decode())
    return out


def resize_taps(in_size, out_size):
    """host half of the pre-processing (no GPU): (start[out+1], src[], w[]) tap lists of one axis"""
    start = np.zeros(out_size + 1, dtype=np.int32)
    cap = 16 * max(in_size, out_size) + 64
    while True:
        src, w = np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.float32)
        n = lib().mars_b200_resize_taps(in_size, out_size, start.ctypes.data, src.ctypes.data, w.ctypes.data, cap)
        if n < 0:
            raise ValueError("resize_taps(%d, %d)" % (in_size, out_size))
        if n <= cap:
            return start, src[:n].copy(), w[:n].copy()
        cap = n


def tile_rois(w, h, tile_w=640, tile_h=640, overlap_w=128, overlap_h=128, with_full=False, frame=0):
    """host only (no GPU): the tile grid of a w x h frame (mars_b200_tile_rois) as a ROI_DTYPE array"""
    n = lib().mars_b200_tile_rois(frame, w, h, tile_w, tile_h, overlap_w, overlap_h, 1 if with_full else 0, None, 0)
    if n < 0:
        raise ValueError("tile_rois(%d, %d, %d, %d, %d, %d)" % (w, h, tile_w, tile_h, overlap_w, overlap_h))
    out = np.zeros(n, dtype=ROI_DTYPE)
    assert lib().mars_b200_tile_rois(frame, w, h, tile_w, tile_h, overlap_w, overlap_h, 1 if with_full else 0, out.ctypes.data, n) == n
    return out


def yuv_coefficients(colour):
    """host half of the NV12 conversion (no GPU): [y0, cy, crv, cgu, cgv, cbu] of a colour variant (YUV_*)"""
    out = np.zeros(6, dtype=np.int32)
    if lib().mars_b200_yuv_coefficients(colour, out.ctypes.data) != 0:
        raise ValueError("yuv_coefficients(%d)" % colour)
    return out


def find_yolo_heads(blob):
    """tensor ids of the three YOLOv5 Detect head convs of a .mars blob in stride order 8 / 16 / 32, or [] (host only, no GPU)"""
    b = bytes(blob)
    ids = (C.c_uint32 * 3)()
    n = lib().mars_b200_find_yolo_heads(b, len(b), ids, 3)
    return [int(v) for v in ids[:n]]


GFL_CENTRE = {"half": 0, "corner": 1}  # MARS_B200_GFL_CENTRE_HALF / _CORNER


def find_gfl_heads(blob, nc=80, reg_max=7):
    """tensor ids of the NanoDet GFL head convs of a .mars blob in stride order 8 / 16 / 32 (/ 64), or [] (host only, no GPU)"""
    b = bytes(blob)
    ids = (C.c_uint32 * 4)()
    n = lib().mars_b200_find_gfl_heads(b, len(b), nc, reg_max, ids, 4)
    return [int(v) for v in ids[:n]]


# ---- post-process on host arrays (runs on the device) ---------------------------------
def parse_output(out_i8, npred, scale, maxd=1000):
    dets = np.zeros(max(maxd, 1), dtype=DET_DTYPE)
    buf = np.ascontiguousarray(out_i8).view(np.int8)
    n = lib().mars_yolo_parse_output(buf.ctypes.data, npred, scale, dets.ctypes.data, maxd)
    return dets[:n].copy()


def nms(dets, thresh=0.45):
    d = np.ascontiguousarray(dets.copy())
    n = lib().mars_yolo_nms(d.ctypes.data, len(d), thresh)
    return d[:max(n, 0)].copy()


def decode_gfl(head, nc, reg_max, scale, stride, net_w, net_h, conf_thresh=0.25, centre="half", dets=None, cnt=0, maxd=1000):
    """GFL decode of one int8 [gh, gw, nc + 4 (reg_max + 1)] head on the device (k_gfl_decode): boxes appended after dets[:cnt]
    (dets: BOX_DTYPE [>= maxd] or None), returns dets[:count]"""
    h = np.ascontiguousarray(head, dtype=np.int8)
    gh, gw, _ = h.shape
    out = np.zeros(maxd, dtype=BOX_DTYPE)
    if dets is not None and cnt:
        out[:cnt] = dets[:cnt]
    code = GFL_CENTRE[centre] if isinstance(centre, str) else int(centre)
    n = lib().mars_b200_decode_gfl(h.ctypes.data, gh, gw, nc, reg_max, scale, stride, code, net_w, net_h, conf_thresh, out.ctypes.data,
                                   cnt, maxd)
    return out[:n].copy()


def nms_boxes(boxes, thresh=0.45):
    d = np.ascontiguousarray(boxes.copy())
    n = lib().mars_yolo_nms_boxes(d.ctypes.data, len(d), thresh)
    return d[:max(n, 0)].copy()
