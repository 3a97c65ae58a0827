"""ctypes binding of the C ABI in include/instance_stixels_b200.h.

The shared library is built in-tree by `__graft_entry__.build()` /
`make -C instance_stixels_b200/csrc`.  There is no fallback: a missing library
or a missing CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ISX_LIB_PATH: a differently tuned build of the same library (kernel A/B runs); there is no other fallback
LIB_PATH = os.environ.get("ISX_LIB_PATH") or os.path.join(_HERE, "libinstance_stixels_b200.so")

# every symbol include/instance_stixels_b200.h declares
EXPORTS = [
    "isx_abi_version", "isx_kernel_launch_count", "isx_last_error", "isx_config_init", "isx_create",
    "isx_destroy", "isx_set_config", "isx_set_disparity_parameters", "isx_set_segmentation_parameters",
    "isx_set_clustering_parameters", "isx_set_weight_parameters", "isx_set_probabilities",
    "isx_set_camera_parameters", "isx_set_model_parameters", "isx_initialize", "isx_finish",
    "isx_is_initialized", "isx_real_cols", "isx_max_sections", "isx_segmentation_elems",
    "isx_set_disparity_image", "isx_input_disparity_device", "isx_set_segmentation",
    "isx_set_road_parameters", "isx_compute", "isx_cluster_instances", "isx_dbscan_fit_host", "isx_instance_capacity", "isx_get_dp_units", "isx_flush",
    "isx_get_instance_stixels",
    "isx_compute_batch_host", "isx_submit_batch_host", "isx_wait_batch_host", "isx_reserve_in_flight", "isx_compute_batch_device", "isx_synchronize", "isx_fetch_batch_results",
    "isx_stream", "isx_tensor_elems", "isx_read_tensor", "isx_set_profiling", "isx_get_stage_times",
    "isx_chunk_frames", "isx_get_chunk_trace", "isx_host_alloc", "isx_host_free",
    # compact results / narrow inputs / frame pool
    "isx_wait_batch_packed", "isx_narrow_segmentation_elems", "isx_compute_batch_host_u16", "isx_submit_batch_host_u16",
    "isx_pool_create", "isx_pool_destroy", "isx_pool_size", "isx_pool_real_cols", "isx_pool_segmentation_elems",
    "isx_pool_compute_host", "isx_pool_last_error", "isx_pool_frames_by_worker",
    # segmentation ingest (SURVEY.md 8f rank 2)
    "isx_set_segmentation_from_cnn_device", "isx_flip_and_pad_batch_device",
    # result images (SURVEY.md 8f rank 3)
    "isx_rasterize_batch_device",
    # device results
    "isx_export_batch_device",
    # road estimation (SURVEY.md 8f rank 1)
    "isx_road_create", "isx_road_destroy", "isx_road_initialize", "isx_road_finish", "isx_road_is_initialized",
    "isx_road_compute_host", "isx_road_compute_device", "isx_road_compute_batch_device", "isx_road_last_error",
    "isx_road_tensor_bytes", "isx_road_read_tensor",
    # device batches with road estimation in stream order
    "isx_compute_batch_device_road",
]


class Config(C.Structure):
    """isx_config == StixelConfig (types.h:30-141)."""
    _fields_ = [
        ("rows", C.c_float), ("cols", C.c_float), ("max_dis", C.c_int32), ("invalid_disparity", C.c_float),
        ("eps", C.c_float), ("min_pts", C.c_int32), ("size_filter", C.c_int32),
        ("n_semantic_classes", C.c_int32), ("n_offset_channels", C.c_int32),
        ("prior_weight", C.c_float), ("segmentation_weight", C.c_float), ("instance_weight", C.c_float),
        ("disparity_weight", C.c_float), ("pairwise", C.c_int32), ("column_step", C.c_int32),
        ("focal", C.c_float), ("baseline", C.c_float), ("camera_center_x", C.c_float),
        ("camera_center_y", C.c_float),
        ("sigma_disparity_object", C.c_float), ("sigma_disparity_ground", C.c_float), ("sigma_sky", C.c_float),
        ("pout", C.c_float), ("pout_sky", C.c_float), ("pord", C.c_float), ("pgrav", C.c_float),
        ("pblg", C.c_float),
        ("pground_given_nexist", C.c_float), ("pobject_given_nexist", C.c_float),
        ("psky_given_nexist", C.c_float), ("pnexist_dis", C.c_float), ("pground", C.c_float),
        ("pobject", C.c_float), ("psky", C.c_float), ("width_margin", C.c_int32),
        ("sigma_camera_tilt", C.c_float), ("sigma_camera_height", C.c_float), ("median_join", C.c_int32),
        ("epsilon", C.c_float), ("range_objects_z", C.c_float), ("road_vdisparity_threshold", C.c_float),
    ]


class FrameMeta(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("rows", "cols", "realcols", "max_sections", "max_dis", "column_step", "semantic_classes")] + \
               [("alpha_ground", C.c_float), ("vhor", C.c_int32)]


class Road(C.Structure):
    _fields_ = [("vhor", C.c_int32), ("camera_tilt", C.c_float), ("camera_height", C.c_float),
                ("alpha_ground", C.c_float)]


class RoadEstimate(C.Structure):
    """isx_road_estimate: what RoadEstimation::Compute leaves in its getters (RoadEstimation.h:46-50)."""
    _fields_ = [("ok", C.c_int32), ("horizon_point", C.c_int32), ("pitch", C.c_float), ("camera_height", C.c_float),
                ("slope", C.c_float), ("rho", C.c_float), ("theta", C.c_float)]


class DeviceResults(C.Structure):
    """isx_device_results: device pointers the export writes (None = not written; frame_offsets is required)."""
    _fields_ = [("sections", C.c_void_p), ("frame_offsets", C.c_void_p), ("column_offsets", C.c_void_p),
                ("labels", C.c_void_p), ("vertices", C.c_void_p), ("frame_errors", C.c_void_p),
                ("capacity", C.c_int32), ("reserved", C.c_int32)]


# numpy views of isx_section (== Section, types.h:186-194) and isx_instance
SECTION_DTYPE = np.dtype([("type", "<i4"), ("vB", "<i4"), ("vT", "<i4"), ("disparity", "<f4"),
                          ("semantic_class", "<i4"), ("cost", "<f4"), ("instance_meanx", "<f4"),
                          ("instance_meany", "<f4")])
INSTANCE_DTYPE = np.dtype([("column", "<i4"), ("index", "<i4"), ("label", "<i4"), ("semantic_class", "<i4")])
PACKED_FRAME_DTYPE = np.dtype([("section_offset", "<i4"), ("section_count", "<i4"), ("instance_offset", "<i4"),
                               ("instance_count", "<i4"), ("error", "<i4"), ("overflow", "<i4"),
                               ("reserved", "<i4", (2,))])
assert SECTION_DTYPE.itemsize == 32 and INSTANCE_DTYPE.itemsize == 16 and PACKED_FRAME_DTYPE.itemsize == 32

ISX_OK = 0
T_JOINED_DISPARITY, T_OBJECT_LUT, T_DISPARITY_PS, T_VALID_PS, T_GROUND_PS, T_SKY_PS, T_COST_TABLE, \
    T_INDEX_TABLE, T_GROUND_TABLES, T_OBJ_COST_LUT, T_OBJECT_DISPARITY_RANGE = range(11)

_lib = None


def _declare(lib):
    H = C.c_void_p
    f, i = C.c_float, C.c_int
    lib.isx_abi_version.restype = i
    lib.isx_kernel_launch_count.restype = C.c_uint64
    lib.isx_last_error.restype = C.c_char_p
    lib.isx_last_error.argtypes = [H]
    lib.isx_config_init.argtypes = [C.POINTER(Config)]
    lib.isx_config_init.restype = None
    lib.isx_create.argtypes = [C.POINTER(H), i]
    lib.isx_destroy.argtypes = [H]
    lib.isx_set_config.argtypes = [H, C.POINTER(Config)]
    lib.isx_set_disparity_parameters.argtypes = [H, i, i, i, f, f, f, f]
    lib.isx_set_segmentation_parameters.argtypes = [H, i, i]
    lib.isx_set_clustering_parameters.argtypes = [H, f, i, i]
    lib.isx_set_weight_parameters.argtypes = [H, f, f, f, f]
    lib.isx_set_probabilities.argtypes = [H] + [f] * 12
    lib.isx_set_camera_parameters.argtypes = [H] + [f] * 6
    lib.isx_set_model_parameters.argtypes = [H, i, i, f, f, i]
    lib.isx_initialize.argtypes = [H, i]
    lib.isx_finish.argtypes = [H]
    lib.isx_is_initialized.argtypes = [H]
    lib.isx_real_cols.argtypes = [H]
    lib.isx_max_sections.argtypes = [H]
    lib.isx_segmentation_elems.argtypes = [H]
    lib.isx_segmentation_elems.restype = C.c_size_t
    lib.isx_set_disparity_image.argtypes = [H, C.c_void_p, C.c_size_t]
    lib.isx_input_disparity_device.argtypes = [H]
    lib.isx_input_disparity_device.restype = C.c_void_p
    lib.isx_set_segmentation.argtypes = [H, C.c_void_p, C.c_size_t]
    lib.isx_set_road_parameters.argtypes = [H, i, f, f, f]
    lib.isx_compute.argtypes = [H, i, C.c_void_p, C.POINTER(FrameMeta), C.c_void_p]
    lib.isx_cluster_instances.argtypes = [H]
    lib.isx_dbscan_fit_host.argtypes = [i, C.c_void_p, i, f, i, C.c_void_p, C.c_void_p]
    lib.isx_get_instance_stixels.argtypes = [H, C.c_void_p, i, C.POINTER(i)]
    lib.isx_compute_batch_host.argtypes = [H, i, i, C.c_void_p, C.c_void_p, C.POINTER(Road), C.c_void_p,
                                           C.c_void_p, i, C.c_void_p]
    lib.isx_submit_batch_host.argtypes = [H, i, i, C.c_void_p, C.c_void_p, C.POINTER(Road), C.c_void_p]
    lib.isx_wait_batch_host.argtypes = [H, C.c_void_p, i, C.c_void_p]
    lib.isx_reserve_in_flight.argtypes = [H, i]
    lib.isx_wait_batch_packed.argtypes = [H] + [C.POINTER(C.c_void_p)] * 4 + [C.POINTER(i)]
    lib.isx_narrow_segmentation_elems.argtypes = [H]
    lib.isx_narrow_segmentation_elems.restype = C.c_size_t
    lib.isx_compute_batch_host_u16.argtypes = [H, i, i, C.c_void_p, f, C.c_void_p, C.POINTER(Road), C.c_void_p,
                                               C.c_void_p, i, C.c_void_p]
    lib.isx_submit_batch_host_u16.argtypes = [H, i, i, C.c_void_p, f, C.c_void_p, C.POINTER(Road), C.c_void_p]
    lib.isx_pool_create.argtypes = [C.POINTER(H), C.POINTER(i), i, C.POINTER(Config), i]
    lib.isx_pool_destroy.argtypes = [H]
    lib.isx_pool_size.argtypes = [H]
    lib.isx_pool_real_cols.argtypes = [H]
    lib.isx_pool_segmentation_elems.argtypes = [H]
    lib.isx_pool_segmentation_elems.restype = C.c_size_t
    lib.isx_pool_compute_host.argtypes = [H, i, i, C.c_void_p, C.c_void_p, C.POINTER(Road), C.c_void_p, C.c_void_p, i,
                                          C.c_void_p]
    lib.isx_pool_last_error.argtypes = [H]
    lib.isx_pool_last_error.restype = C.c_char_p
    lib.isx_pool_frames_by_worker.argtypes = [H, C.POINTER(C.c_int), i]
    lib.isx_compute_batch_device.argtypes = [H, i, i, C.c_void_p, C.c_void_p, C.POINTER(Road)]
    lib.isx_synchronize.argtypes = [H]
    lib.isx_flush.argtypes = [H]
    lib.isx_fetch_batch_results.argtypes = [H, i, C.c_void_p, C.c_void_p, i, C.c_void_p]
    lib.isx_stream.argtypes = [H]
    lib.isx_stream.restype = C.c_uint64
    lib.isx_tensor_elems.argtypes = [H, i]
    lib.isx_tensor_elems.restype = C.c_size_t
    lib.isx_read_tensor.argtypes = [H, i, i, C.c_void_p, C.c_size_t]
    lib.isx_set_profiling.argtypes = [H, i]
    lib.isx_get_stage_times.argtypes = [H, C.POINTER(C.c_double), C.POINTER(C.c_long), i, i]
    lib.isx_chunk_frames.argtypes = [H]
    lib.isx_host_alloc.argtypes = [C.c_size_t]
    lib.isx_host_alloc.restype = C.c_void_p
    lib.isx_host_free.argtypes = [C.c_void_p]
    lib.isx_host_free.restype = None
    lib.isx_get_chunk_trace.argtypes = [H, C.POINTER(C.c_double), i]
    lib.isx_get_dp_units.argtypes = [H, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    lib.isx_instance_capacity.argtypes = [H]
    lib.isx_set_segmentation_from_cnn_device.argtypes = [H, C.c_void_p, i, i]
    lib.isx_flip_and_pad_batch_device.argtypes = [H, i, C.c_void_p, i, i, C.c_void_p]
    lib.isx_rasterize_batch_device.argtypes = [H, i, i, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.isx_export_batch_device.argtypes = [H, i, i, C.POINTER(DeviceResults)]
    lib.isx_road_create.argtypes = [C.POINTER(H), i]
    lib.isx_road_destroy.argtypes = [H]
    lib.isx_road_destroy.restype = None
    lib.isx_road_initialize.argtypes = [H, f, f, f, i, i, i, f, i]
    lib.isx_road_finish.argtypes = [H]
    lib.isx_road_is_initialized.argtypes = [H]
    lib.isx_road_compute_host.argtypes = [H, C.c_void_p, C.c_size_t, C.POINTER(RoadEstimate)]
    lib.isx_road_compute_device.argtypes = [H, C.c_void_p, C.POINTER(RoadEstimate)]
    lib.isx_road_compute_batch_device.argtypes = [H, i, C.c_void_p, C.POINTER(RoadEstimate)]
    lib.isx_road_last_error.argtypes = [H]
    lib.isx_road_last_error.restype = C.c_char_p
    lib.isx_road_tensor_bytes.argtypes = [H, i]
    lib.isx_road_tensor_bytes.restype = C.c_size_t
    lib.isx_road_read_tensor.argtypes = [H, i, i, C.c_void_p, C.c_size_t]
    lib.isx_compute_batch_device_road.argtypes = [H, H, i, i, C.c_void_p, C.c_void_p, C.POINTER(Road), C.c_void_p,
                                                  C.c_void_p]


def load():
    """Load the CUDA library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the stixel path)")
        lib = C.CDLL(LIB_PATH)
        _declare(lib)
        _lib = lib
    return _lib
