"""Python mirror of the reference's `Stixels` class over the C ABI.

Method names, argument meaning and error behaviour follow
InstanceStixels/include/InstanceStixels/Stixels.hpp:40-96 so that tests read
like the call sequence of apps/run_cityscapes.cu:335-449.  The product path is
the CUDA library; nothing here computes.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any, Optional, Sequence

import numpy as np

from . import _lib as L


class StixelsError(RuntimeError):
    pass


class InvalidArgument(ValueError):
    """Where the reference throws std::invalid_argument (Stixels.cu:292-313, 685-687)."""


def StixelConfig(**fields) -> L.Config:
    """`StixelConfig` with the reference's defaults (types.h:30-141) + overrides."""
    lib = L.load()
    cfg = L.Config()
    lib.isx_config_init(C.byref(cfg))
    names = {n for n, _ in L.Config._fields_}
    for k, v in fields.items():
        if k not in names:
            raise AttributeError(f"StixelConfig has no field {k!r}")
        setattr(cfg, k, int(v) if isinstance(v, bool) else v)
    return cfg


def _roads(roads: Sequence[dict]):
    arr = (L.Road * len(roads))()
    for i, r in enumerate(roads):
        arr[i] = L.Road(int(r["vhor"]), float(r["camera_tilt"]), float(r["camera_height"]),
                        float(r["alpha_ground"]))
    return arr


class StixelsData:
    """types.h:196-205."""

    def __init__(self, sections: np.ndarray, meta: L.FrameMeta):
        self.sections = sections
        for n, _ in L.FrameMeta._fields_:
            setattr(self, n, getattr(meta, n))


def _f32():
    import torch
    return torch.float32


@dataclass
class DeviceRoadEstimates:
    """isx_road_estimate records on the device: `data` is the int32 [n, 7] tensor, the properties are its columns."""
    data: Any

    ok = property(lambda self: self.data[:, 0])
    horizon_point = property(lambda self: self.data[:, 1])
    pitch = property(lambda self: self.data[:, 2].view(_f32()))
    camera_height = property(lambda self: self.data[:, 3].view(_f32()))
    slope = property(lambda self: self.data[:, 4].view(_f32()))
    rho = property(lambda self: self.data[:, 5].view(_f32()))
    theta = property(lambda self: self.data[:, 6].view(_f32()))


@dataclass
class DeviceRoads:
    """isx_road records on the device (the SetRoadParameters arguments of every frame): `data` is int32 [n, 4]."""
    data: Any

    vhor = property(lambda self: self.data[:, 0])
    camera_tilt = property(lambda self: self.data[:, 1].view(_f32()))
    camera_height = property(lambda self: self.data[:, 2].view(_f32()))
    alpha_ground = property(lambda self: self.data[:, 3].view(_f32()))


@dataclass
class DeviceStixels:
    """Torch tensors of Stixels.ComputeBatchTensors (the isx_device_results layout).  `sections` is the int32
    [capacity, 8] view of the Sections; frame f owns rows [frame_offsets[f], frame_offsets[f+1]); `vertices` is
    [capacity, 4, 3] or None.  With road estimation on the device (road=), `road_estimates` holds what the
    estimation returned for every frame and `roads` the road every frame was computed with."""
    sections: Any
    frame_offsets: Any
    column_offsets: Any
    labels: Any
    vertices: Any
    frame_errors: Any
    road_estimates: Optional[DeviceRoadEstimates] = None
    roads: Optional[DeviceRoads] = None

    # typed columns of `sections` (isx_section)
    @property
    def type(self):
        return self.sections[:, 0]

    @property
    def vB(self):
        return self.sections[:, 1]

    @property
    def vT(self):
        return self.sections[:, 2]

    @property
    def disparity(self):
        return self.sections[:, 3].view(self._f32())

    @property
    def semantic_class(self):
        return self.sections[:, 4]

    @property
    def cost(self):
        return self.sections[:, 5].view(self._f32())

    @property
    def instance_meanx(self):
        return self.sections[:, 6].view(self._f32())

    @property
    def instance_meany(self):
        return self.sections[:, 7].view(self._f32())

    @staticmethod
    def _f32():
        import torch
        return torch.float32


class Stixels:
    def __init__(self, device: int = 0):
        self._lib = L.load()
        self._h = C.c_void_p()
        self._check(self._lib.isx_create(C.byref(self._h), device), None)
        self._device = device
        self._pairwise = False

    # -- plumbing ---------------------------------------------------------
    def _check(self, rc, h="self"):
        if rc == L.ISX_OK:
            return
        msg = self._lib.isx_last_error(self._h if h == "self" else None)
        msg = msg.decode() if msg else ""
        if rc == -1:
            raise InvalidArgument(msg)
        raise StixelsError(f"isx error {rc}: {msg}")

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.isx_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # -- reference API ----------------------------------------------------
    def SetConfig(self, config: L.Config):
        self._check(self._lib.isx_set_config(self._h, C.byref(config)))
        self._pairwise = bool(config.pairwise)
        self._cols = int(config.cols)

    def Initialize(self, max_batch: int = 1):
        self._check(self._lib.isx_initialize(self._h, max_batch))

    def Finish(self):
        self._check(self._lib.isx_finish(self._h))

    def IsInitialized(self) -> bool:
        return bool(self._lib.isx_is_initialized(self._h))

    def GetRealCols(self) -> int:
        return self._lib.isx_real_cols(self._h)

    def GetMaxSections(self) -> int:
        return self._lib.isx_max_sections(self._h)

    def segmentation_elems(self) -> int:
        return self._lib.isx_segmentation_elems(self._h)

    def SetDisparityImage(self, disp_im: np.ndarray):
        a = np.ascontiguousarray(disp_im, dtype=np.float32)
        self._keep_disp = a
        self._check(self._lib.isx_set_disparity_image(self._h, a.ctypes.data, a.size))

    def GetInputDisparityImageOnDevice(self) -> int:
        return self._lib.isx_input_disparity_device(self._h)

    def SetSegmentation(self, segmentation: np.ndarray):
        a = np.ascontiguousarray(segmentation, dtype=np.int32)
        self._keep_seg = a
        self._check(self._lib.isx_set_segmentation(self._h, a.ctypes.data, a.size))

    def SetSegmentationFromCNN(self, d_cnn: int, cnn_rows: int, cnn_cols: int):
        """FlipAndPad on the device (wrappers.py:35-61): plain CNN output float [21][rows/8][cols/8] (device
        pointer) -> the tensor SetSegmentation uploads."""
        self._check(self._lib.isx_set_segmentation_from_cnn_device(self._h, d_cnn, cnn_rows, cnn_cols))

    def FlipAndPadBatchDevice(self, n: int, d_cnn: int, cnn_rows: int, cnn_cols: int, d_segmentation: int):
        """n CNN outputs -> the segmentation layout ComputeBatchDevice takes; asynchronous."""
        self._check(self._lib.isx_flip_and_pad_batch_device(self._h, n, d_cnn, cnn_rows, cnn_cols, d_segmentation))

    def RasterizeBatchDevice(self, first: int, n: int, d_label_ids: int = 0, d_instance_ids: int = 0,
                             d_disparity: int = 0):
        """Stixels of frames [first, first+n) of the last batch -> label-id / instance-id / disparity images on
        the device (clustering_visualization.py:118-142, 397-409); pointers may be 0."""
        self._check(self._lib.isx_rasterize_batch_device(self._h, first, n, d_label_ids or None,
                                                         d_instance_ids or None, d_disparity or None))

    def ExportBatchDevice(self, first: int, n: int, frame_offsets: int, sections: int = 0, column_offsets: int = 0,
                          labels: int = 0, vertices: int = 0, frame_errors: int = 0, capacity: int = 0):
        """Stixels of frames [first, first+n) of the last batch into caller device buffers (raw pointers, 0 = not
        written): frame-ordered CSR Sections, offsets, instance labels (-2 outside GetInstanceStixels) and
        Get3DVertices per stixel; `capacity` counts stixels.  Asynchronous on stream()."""
        out = L.DeviceResults(sections or None, frame_offsets or None, column_offsets or None, labels or None,
                              vertices or None, frame_errors or None, capacity, 0)
        self._check(self._lib.isx_export_batch_device(self._h, first, n, C.byref(out)))

    def ComputeBatchTensors(self, pairwise: bool, disparity, roads: Optional[Sequence[dict]] = None,
                            segmentation=None, cnn=None, vertices: bool = False, capacity: Optional[int] = None,
                            road: Optional["RoadEstimation"] = None, fallback: Optional[dict] = None) -> "DeviceStixels":
        """CUDA torch tensors in, torch tensors out, no host synchronisation: `disparity` float32 [n][rows][cols]
        and either `segmentation` int32 in the library layout [n][realcols][21][rows_power2_segmentation] or `cnn`
        float32 [n][21][rows/8][cols/8] (run through FlipAndPadBatchDevice).  The library's stream waits for the
        current torch stream, and the current torch stream waits for the results.  `capacity` (stixels) defaults
        to the worst case n * realcols * 200.
        The road of every frame: either `roads` (one dict per frame) or `road`, a RoadEstimation that estimates it
        on the device from the frame's disparity (ComputeBatchDeviceRoad; `fallback` as there).  With `road`, the
        result also carries `road_estimates` and `roads`."""
        import torch
        if (roads is None) == (road is None):
            raise InvalidArgument("pass exactly one of roads= and road=")
        if fallback is not None and road is None:
            raise InvalidArgument("fallback= goes with road=")
        if (segmentation is None) == (cnn is None):
            raise InvalidArgument("pass exactly one of segmentation= and cnn=")
        if not (disparity.is_cuda and disparity.dtype == torch.float32 and disparity.is_contiguous()):
            raise InvalidArgument("disparity must be a contiguous float32 CUDA tensor")
        n = len(roads) if roads is not None else disparity.numel() // self._frame_pixels()
        if n < 1:
            raise InvalidArgument("disparity must hold n >= 1 frames of rows*cols")
        inputs = [disparity]
        dev = disparity.device
        if dev.index != self._device:
            raise InvalidArgument(f"the tensors are on {dev}, the handle computes on cuda:{self._device}")
        C_ = self.GetRealCols()
        if cnn is not None:
            if not (cnn.device == dev and cnn.dtype == torch.float32 and cnn.is_contiguous() and cnn.dim() == 4
                    and cnn.shape[0] == n):
                raise InvalidArgument("cnn must be a contiguous float32 tensor [n][21][rows/8][cols/8] on the handle's device")
            inputs.append(cnn)
            segmentation = torch.empty(n * self.segmentation_elems(), dtype=torch.int32, device=dev)
        elif not (segmentation.device == dev and segmentation.dtype == torch.int32 and segmentation.is_contiguous()
                  and segmentation.numel() == n * self.segmentation_elems()):
            raise InvalidArgument("segmentation must be a contiguous int32 tensor in the library layout on the handle's device")
        inputs.append(segmentation)
        if disparity.numel() != n * self._frame_pixels():
            raise InvalidArgument("disparity must hold n frames of rows*cols")
        cap = n * C_ * self.GetMaxSections() if capacity is None else int(capacity)
        out = DeviceStixels(
            sections=torch.empty((cap, 8), dtype=torch.int32, device=dev),
            frame_offsets=torch.empty(n + 1, dtype=torch.int32, device=dev),
            column_offsets=torch.empty(n * C_ + 1, dtype=torch.int32, device=dev),
            labels=torch.empty(cap, dtype=torch.int32, device=dev),
            vertices=torch.empty((cap, 4, 3), dtype=torch.float32, device=dev) if vertices else None,
            frame_errors=torch.empty(n, dtype=torch.int32, device=dev))
        if road is not None:
            out.road_estimates = DeviceRoadEstimates(torch.empty((n, 7), dtype=torch.int32, device=dev))
            out.roads = DeviceRoads(torch.empty((n, 4), dtype=torch.int32, device=dev))
        current = torch.cuda.current_stream(dev)
        ext = torch.cuda.ExternalStream(self.stream(), device=dev)
        # the inputs and the outputs allocated above are ready on the current stream
        ready = torch.cuda.Event()
        ready.record(current)
        ext.wait_event(ready)
        for t in inputs:
            t.record_stream(ext)   # read on the library's stream: not reused before that work is done
        if cnn is not None:
            self.FlipAndPadBatchDevice(n, cnn.data_ptr(), cnn.shape[2], cnn.shape[3], segmentation.data_ptr())
        if road is None:
            self.ComputeBatchDevice(pairwise, n, disparity.data_ptr(), segmentation.data_ptr(), roads)
        else:
            self.ComputeBatchDeviceRoad(road, pairwise, n, disparity.data_ptr(), segmentation.data_ptr(), fallback,
                                        out.road_estimates.data.data_ptr(), out.roads.data.data_ptr())
        self.ExportBatchDevice(0, n, out.frame_offsets.data_ptr(), sections=out.sections.data_ptr(),
                               column_offsets=out.column_offsets.data_ptr(), labels=out.labels.data_ptr(),
                               vertices=out.vertices.data_ptr() if vertices else 0,
                               frame_errors=out.frame_errors.data_ptr(), capacity=cap)
        done = torch.cuda.Event()
        done.record(ext)
        current.wait_event(done)
        return out

    def SetRoadParameters(self, vhor: int, camera_tilt: float, camera_height: float, alpha_ground: float):
        self._check(self._lib.isx_set_road_parameters(self._h, vhor, camera_tilt, camera_height, alpha_ground))

    def SetSegmentationParameters(self, classes, instance_channels):
        self._check(self._lib.isx_set_segmentation_parameters(self._h, classes, instance_channels))

    def SetClusteringParameters(self, eps, min_pts, size_filter):
        self._check(self._lib.isx_set_clustering_parameters(self._h, eps, min_pts, size_filter))

    def SetWeightParameters(self, prior_weight, disparity_weight, segmentation_weight, instance_weight):
        self._check(self._lib.isx_set_weight_parameters(self._h, prior_weight, disparity_weight,
                                                        segmentation_weight, instance_weight))

    def SetProbabilities(self, *a):
        self._check(self._lib.isx_set_probabilities(self._h, *a))

    def SetCameraParameters(self, focal, baseline, sigma_camera_tilt, sigma_camera_height,
                            camera_center_x=-1.0, camera_center_y=-1.0):
        self._check(self._lib.isx_set_camera_parameters(self._h, focal, baseline, sigma_camera_tilt,
                                                        sigma_camera_height, camera_center_x, camera_center_y))

    def SetDisparityParameters(self, rows, cols, max_dis, invalid_disparity, sigma_disparity_object,
                               sigma_disparity_ground, sigma_sky):
        self._check(self._lib.isx_set_disparity_parameters(self._h, rows, cols, max_dis, invalid_disparity,
                                                           sigma_disparity_object, sigma_disparity_ground,
                                                           sigma_sky))

    def SetModelParameters(self, column_step, median_join, epsilon, range_objects_z, width_margin):
        self._check(self._lib.isx_set_model_parameters(self._h, column_step, int(median_join), epsilon,
                                                       range_objects_z, width_margin))

    def Compute(self, pairwise: bool, d_segmentation_local: Optional[int] = None,
                sections_out: Optional[np.ndarray] = None) -> StixelsData:
        """Returns the StixelsData the reference fills through its out-parameter.  `sections_out`: an optional
        caller-owned buffer of realcols*max_sections Sections (e.g. pinned) to fill instead of a new array."""
        n = self.GetRealCols() * self.GetMaxSections()
        if sections_out is not None:
            sections = sections_out.reshape(-1)
            if sections.dtype != L.SECTION_DTYPE or sections.size != n or not sections.flags.c_contiguous:
                raise InvalidArgument("sections_out must hold realcols*max_sections contiguous Sections")
        else:
            sections = np.zeros(n, dtype=L.SECTION_DTYPE)
        meta = L.FrameMeta()
        self._check(self._lib.isx_compute(self._h, int(pairwise), sections.ctypes.data, C.byref(meta),
                                          d_segmentation_local))
        return StixelsData(sections.reshape(self.GetRealCols(), self.GetMaxSections()), meta)

    def ClusterInstances(self):
        self._check(self._lib.isx_cluster_instances(self._h))

    def GetInstanceStixels(self) -> dict:
        """{(column, index): label} like the reference's std::map (Stixels.cu:744-776)."""
        inst = self.instance_records()
        return dict(zip(zip(inst["column"].tolist(), inst["index"].tolist()), inst["label"].tolist()))

    def instance_records(self) -> np.ndarray:
        n = C.c_int(0)
        self._check(self._lib.isx_get_instance_stixels(self._h, None, 0, C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=L.INSTANCE_DTYPE)
        self._check(self._lib.isx_get_instance_stixels(self._h, out.ctypes.data, n.value, C.byref(n)))
        return out[:n.value]

    # -- batched extensions (no reference counterpart) ---------------------
    def ComputeBatch(self, pairwise: bool, disparity: np.ndarray, segmentation: np.ndarray,
                     roads: Sequence[dict], sections_out: Optional[np.ndarray] = None,
                     want_instances: bool = True):
        """Host buffers in, host results out (H2D/D2H inside). Returns (sections, instances, offsets)."""
        n = len(roads)
        disparity = np.ascontiguousarray(disparity, dtype=np.float32)
        segmentation = np.ascontiguousarray(segmentation, dtype=np.int32)
        C_, S = self.GetRealCols(), self.GetMaxSections()
        if sections_out is None:
            sections_out = np.zeros((n, C_, S), dtype=L.SECTION_DTYPE)
        inst, offs, cap = self._instance_buffers(n) if want_instances else (None, None, 0)
        self._check(self._lib.isx_compute_batch_host(
            self._h, int(pairwise), n, disparity.ctypes.data, segmentation.ctypes.data, _roads(roads),
            sections_out.ctypes.data, inst.ctypes.data if want_instances else None,
            cap, offs.ctypes.data if want_instances else None))
        if not want_instances:
            return sections_out, np.zeros(0, dtype=L.INSTANCE_DTYPE), np.zeros(n + 1, dtype=np.int32)
        return sections_out, inst[:offs[n]].copy(), offs.copy()

    def SubmitBatch(self, pairwise: bool, disparity: np.ndarray, segmentation: np.ndarray, roads: Sequence[dict],
                    sections_out: np.ndarray):
        """Asynchronous ComputeBatch: enqueue one batch (host buffers, which must stay alive and unchanged until
        the matching WaitBatch) and return.  At most three batches in flight."""
        n = len(roads)
        if disparity.dtype != np.float32 or segmentation.dtype != np.int32 or \
                not disparity.flags.c_contiguous or not segmentation.flags.c_contiguous:
            raise InvalidArgument("SubmitBatch needs C-contiguous float32 / int32 arrays (no hidden copies)")
        self._check(self._lib.isx_submit_batch_host(self._h, int(pairwise), n, disparity.ctypes.data,
                                                    segmentation.ctypes.data, _roads(roads),
                                                    sections_out.ctypes.data if sections_out is not None else None))
        self._in_flight = getattr(self, "_in_flight", [])
        self._in_flight.append((n, disparity, segmentation, sections_out))

    def narrow_segmentation_elems(self) -> int:
        return self._lib.isx_narrow_segmentation_elems(self._h)

    def ComputeBatchU16(self, pairwise: bool, disparity_u16: np.ndarray, disparity_scale: float,
                        segmentation_i16: np.ndarray, roads: Sequence[dict],
                        sections_out: Optional[np.ndarray] = None):
        """ComputeBatch with narrow host inputs: uint16 disparity (value = u16 * disparity_scale, e.g. a 16-bit
        disparity PNG with 1/256) and int16 segmentation [n][C][21][ceil(rows/8)] without the zero padding."""
        n = len(roads)
        d = np.ascontiguousarray(disparity_u16, dtype=np.uint16)
        g = np.ascontiguousarray(segmentation_i16, dtype=np.int16)
        if g.size != n * self.narrow_segmentation_elems() or d.size != n * self._frame_pixels():
            raise InvalidArgument("ComputeBatchU16: wrong input size")
        C_, S = self.GetRealCols(), self.GetMaxSections()
        if sections_out is None:
            sections_out = np.zeros((n, C_, S), dtype=L.SECTION_DTYPE)
        inst, offs, cap = self._instance_buffers(n)
        self._check(self._lib.isx_compute_batch_host_u16(
            self._h, int(pairwise), n, d.ctypes.data, disparity_scale, g.ctypes.data, _roads(roads),
            sections_out.ctypes.data, inst.ctypes.data, cap, offs.ctypes.data))
        return sections_out, inst[:offs[n]].copy(), offs.copy()

    def SubmitBatchU16(self, pairwise: bool, disparity_u16: np.ndarray, disparity_scale: float,
                       segmentation_i16: np.ndarray, roads: Sequence[dict], sections_out: Optional[np.ndarray]):
        """Asynchronous ComputeBatchU16 (see SubmitBatch)."""
        n = len(roads)
        if disparity_u16.dtype != np.uint16 or segmentation_i16.dtype != np.int16 or \
                not disparity_u16.flags.c_contiguous or not segmentation_i16.flags.c_contiguous:
            raise InvalidArgument("SubmitBatchU16 needs C-contiguous uint16 / int16 arrays (no hidden copies)")
        self._check(self._lib.isx_submit_batch_host_u16(
            self._h, int(pairwise), n, disparity_u16.ctypes.data, disparity_scale, segmentation_i16.ctypes.data,
            _roads(roads), sections_out.ctypes.data if sections_out is not None else None))
        self._in_flight = getattr(self, "_in_flight", [])
        self._in_flight.append((n, disparity_u16, segmentation_i16, sections_out))

    def _frame_pixels(self) -> int:
        rows = self._lib.isx_tensor_elems(self._h, L.T_JOINED_DISPARITY) // self.GetRealCols()
        return rows * self._cols

    def WaitBatchPacked(self):
        """Wait for the oldest submitted batch and return its packed results WITHOUT expanding them: views of the
        pinned arrays the device wrote (valid until the second SubmitBatch after this call):
        (sections [total], counts [n][C], instances [total], frames [n] of PACKED_FRAME_DTYPE)."""
        if not getattr(self, "_in_flight", None):
            raise InvalidArgument("no submitted batch is in flight")
        self._in_flight.pop(0)
        ps, pc, pi, pf = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        n = C.c_int(0)
        self._check(self._lib.isx_wait_batch_packed(self._h, C.byref(ps), C.byref(pc), C.byref(pi), C.byref(pf),
                                                    C.byref(n)))
        n = n.value
        C_ = self.GetRealCols()

        def view(ptr, count, dtype):
            if count == 0:
                return np.zeros(0, dtype=dtype)
            buf = (C.c_char * (count * np.dtype(dtype).itemsize)).from_address(ptr.value)
            return np.frombuffer(buf, dtype=dtype, count=count)

        frames = view(pf, n, L.PACKED_FRAME_DTYPE)
        nsec = int((frames["section_offset"] + frames["section_count"]).max()) if n else 0
        ninst = int((frames["instance_offset"] + frames["instance_count"]).max()) if n else 0
        return (view(ps, nsec, L.SECTION_DTYPE), view(pc, n * C_, np.int32).reshape(n, C_),
                view(pi, ninst, L.INSTANCE_DTYPE), frames)

    def WaitBatch(self, want_instances: bool = True):
        """Wait for the oldest submitted batch; returns (sections, instances, offsets) like ComputeBatch."""
        if not getattr(self, "_in_flight", None):
            raise InvalidArgument("no submitted batch is in flight")
        n, _, _, sections_out = self._in_flight.pop(0)
        inst, offs, cap = self._instance_buffers(n) if want_instances else (None, None, 0)
        self._check(self._lib.isx_wait_batch_host(self._h, inst.ctypes.data if want_instances else None, cap,
                                                  offs.ctypes.data if want_instances else None))
        if not want_instances:
            return sections_out, np.zeros(0, dtype=L.INSTANCE_DTYPE), np.zeros(n + 1, dtype=np.int32)
        return sections_out, inst[:offs[n]].copy(), offs.copy()

    def _instance_buffers(self, n: int):
        """Reusable result buffers for the packed instance records of a batch of n frames (every stixel of a frame
        can be an instance stixel: isx_instance_capacity() records per frame)."""
        cap = self.instance_capacity() * n
        cached = getattr(self, "_inst_cache", None)
        if cached is None or cached[2] != cap:
            cached = (np.empty(cap, dtype=L.INSTANCE_DTYPE), np.zeros(n + 1, dtype=np.int32), cap)
            self._inst_cache = cached
        return cached

    def ComputeBatchDevice(self, pairwise: bool, n: int, d_disparity: int, d_segmentation: int,
                           roads: Sequence[dict]):
        """Device pointers in, results stay on the device; asynchronous."""
        self._check(self._lib.isx_compute_batch_device(self._h, int(pairwise), n, d_disparity, d_segmentation,
                                                       _roads(roads)))

    def ComputeBatchDeviceRoad(self, road: "RoadEstimation", pairwise: bool, n: int, d_disparity: int,
                               d_segmentation: int, fallback: Optional[dict] = None, d_estimates: int = 0,
                               d_roads: int = 0):
        """ComputeBatchDevice with the road of every frame estimated on the device by `road` (a RoadEstimation
        initialised with the same rows, cols and max_dis), in stream order: asynchronous, no host round trip.  A frame
        without an accepted line keeps the last accepted estimate; before the first, `fallback` (a road dict) is
        used.  fallback=None continues from the state the previous call on `road` left.  d_estimates [n] /
        d_roads [n] (device pointers, 0 = not written) receive the estimates and the roads used."""
        fb = C.byref(_roads([fallback])[0]) if fallback is not None else None
        self._check(self._lib.isx_compute_batch_device_road(self._h, road.handle(), int(pairwise), n, d_disparity,
                                                            d_segmentation, fb, d_estimates or None, d_roads or None))

    def Flush(self):
        """Order the results of every enqueued batch before later work on stream(); asynchronous."""
        self._check(self._lib.isx_flush(self._h))

    def Synchronize(self):
        self._check(self._lib.isx_synchronize(self._h))

    def FetchBatchResults(self, n: int, want_instances: bool = True):
        C_, S = self.GetRealCols(), self.GetMaxSections()
        sections = np.zeros((n, C_, S), dtype=L.SECTION_DTYPE)
        inst, offs, cap = self._instance_buffers(n) if want_instances else (None, None, 0)
        self._check(self._lib.isx_fetch_batch_results(
            self._h, n, sections.ctypes.data, inst.ctypes.data if want_instances else None,
            cap, offs.ctypes.data if want_instances else None))
        if not want_instances:
            return sections, np.zeros(0, dtype=L.INSTANCE_DTYPE), np.zeros(n + 1, dtype=np.int32)
        return sections, inst[:offs[n]].copy(), offs.copy()

    STAGES = ("join", "frame_tables", "column_tables", "dp", "backtrack", "grouping")

    def set_profiling(self, enable: bool):
        self._check(self._lib.isx_set_profiling(self._h, int(enable)))

    def stage_times(self, reset: bool = True) -> dict:
        """{stage: (total_ms, launches)} measured with CUDA events on the library's stream."""
        ms = (C.c_double * 6)()
        ch = (C.c_long * 6)()
        self._check(self._lib.isx_get_stage_times(self._h, ms, ch, 6, int(reset)))
        return {n: (ms[i], ch[i]) for i, n in enumerate(self.STAGES)}

    def ReserveInFlight(self, batches: int):
        """Allocate the result arrays of `batches` (1 .. 3) batches in flight now instead of inside the first
        submits (isx_reserve_in_flight)."""
        self._check(self._lib.isx_reserve_in_flight(self._h, batches))

    def chunk_frames(self) -> int:
        return self._lib.isx_chunk_frames(self._h)

    def dp_units(self):
        """(evaluated, total) 32 x 32-cell units of the DP since Initialize (the unary DP prunes)."""
        ev, tot = C.c_ulonglong(0), C.c_ulonglong(0)
        self._check(self._lib.isx_get_dp_units(self._h, C.byref(ev), C.byref(tot)))
        return ev.value, tot.value

    def instance_capacity(self) -> int:
        return self._lib.isx_instance_capacity(self._h)

    def stream(self) -> int:
        return self._lib.isx_stream(self._h)

    def read_tensor(self, tensor: int, frame: int = 0) -> np.ndarray:
        n = self._lib.isx_tensor_elems(self._h, tensor)
        out = np.zeros(n, dtype=np.int32 if tensor == L.T_INDEX_TABLE else np.float32)
        self._check(self._lib.isx_read_tensor(self._h, tensor, frame, out.ctypes.data, out.nbytes))
        return out


class RoadEstimation:
    """Python mirror of the reference's `RoadEstimation` class (RoadEstimation.h:31-93) over the C ABI:
    Initialize / Finish / Compute / GetCameraHeight / GetPitch / GetSlope / GetHorizonPoint / IsInitialized."""

    def __init__(self, device: int = 0):
        self._lib = L.load()
        self._h = C.c_void_p()
        rc = self._lib.isx_road_create(C.byref(self._h), device)
        if rc != L.ISX_OK:
            raise StixelsError(f"isx_road_create: {self._lib.isx_road_last_error(None).decode()} ({rc})")
        self._est = L.RoadEstimate()
        self._shape = None

    def _check(self, rc):
        if rc != L.ISX_OK:
            msg = self._lib.isx_road_last_error(self._h).decode()
            raise (InvalidArgument if rc == -1 else StixelsError)(f"{msg} ({rc})")

    def __del__(self):
        try:
            if self._h:
                self._lib.isx_road_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def Initialize(self, camera_center_y: float, baseline: float, focal: float, rows: int, cols: int, max_dis: int,
                   road_vdisparity_threshold: float = 0.2, max_batch: int = 1):
        self._check(self._lib.isx_road_initialize(self._h, camera_center_y, baseline, focal, rows, cols, max_dis,
                                                  road_vdisparity_threshold, max_batch))
        self._shape = (rows, cols, max_dis, max_batch)

    def Finish(self):
        self._check(self._lib.isx_road_finish(self._h))

    def IsInitialized(self) -> bool:
        return bool(self._lib.isx_road_is_initialized(self._h))

    def Compute(self, im) -> bool:
        """`im`: host image (numpy, [rows][cols] float32) or a device pointer (int), like the two overloads."""
        if isinstance(im, int):
            self._check(self._lib.isx_road_compute_device(self._h, im, C.byref(self._est)))
        else:
            im = np.ascontiguousarray(im, dtype=np.float32)
            self._check(self._lib.isx_road_compute_host(self._h, im.ctypes.data, im.size, C.byref(self._est)))
        return bool(self._est.ok)

    def ComputeBatchDevice(self, n: int, d_disparity: int):
        """Extension: n device-resident frames -> list of dicts ready for SetRoadParameters / ComputeBatch."""
        est = (L.RoadEstimate * n)()
        self._check(self._lib.isx_road_compute_batch_device(self._h, n, d_disparity, est))
        return [dict(ok=bool(e.ok), vhor=e.horizon_point, camera_tilt=e.pitch, camera_height=e.camera_height,
                     alpha_ground=e.slope, rho=e.rho, theta=e.theta) for e in est]

    def handle(self):
        """The isx_road_handle, for the C entry points (isx_compute_batch_device_road)."""
        return self._h

    def GetCameraHeight(self) -> float:
        return self._est.camera_height

    def GetPitch(self) -> float:
        return self._est.pitch

    def GetSlope(self) -> float:
        return self._est.slope

    def GetHorizonPoint(self) -> int:
        return self._est.horizon_point

    def line(self):
        return self._est.rho, self._est.theta

    def read_tensor(self, tensor: int, frame: int = 0) -> np.ndarray:
        rows, cols, max_dis, _ = self._shape
        nbytes = self._lib.isx_road_tensor_bytes(self._h, tensor)
        out = np.zeros(nbytes, dtype=np.uint8)
        self._check(self._lib.isx_road_read_tensor(self._h, tensor, frame, out.ctypes.data, nbytes))
        if tensor == 0:
            return out.view(np.int32).reshape(rows, max_dis)
        if tensor == 1:
            return out.reshape(rows, max_dis)
        return out.view(np.int32).reshape(-1, 2 * (rows + max_dis) + 3)


def dbscan_fit(xy: np.ndarray, eps: float, min_pts: int, core_candidates: np.ndarray, device: int = 0) -> np.ndarray:
    """The grouping step on one point set, i.e. the reference's
    `ML::dbscanFit(handle, X, n, 2, eps, min_pts, labels, 0, false, core_candidates)` (Stixels.cu:660-666)."""
    lib = L.load()
    xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1, 2)
    cand = np.ascontiguousarray(core_candidates, dtype=np.uint8)
    if len(cand) != len(xy):
        raise InvalidArgument("core_candidates must have one entry per point")
    labels = np.full(len(xy), -1, dtype=np.int32)
    rc = lib.isx_dbscan_fit_host(device, xy.ctypes.data, len(xy), eps, min_pts, cand.ctypes.data, labels.ctypes.data)
    if rc != L.ISX_OK:
        raise StixelsError(f"isx_dbscan_fit_host: {lib.isx_last_error(None).decode()} ({rc})")
    return labels


class StixelsPool:
    """One context + host worker thread per GPU in this process (isx_pool_*): frames of a call are sharded into
    contiguous blocks, frame f -> worker f*G/n, and streamed through the submit/wait pipeline of every context."""

    def __init__(self, config: L.Config, devices: Sequence[int], max_batch: int = 64):
        self._lib = L.load()
        self._p = C.c_void_p()
        devs = (C.c_int * len(devices))(*devices)
        rc = self._lib.isx_pool_create(C.byref(self._p), devs, len(devices), C.byref(config), max_batch)
        if rc != L.ISX_OK:
            raise StixelsError(f"isx_pool_create: {self._lib.isx_pool_last_error(None).decode()} ({rc})")
        self._inst_cap = int(config.cols) // int(config.column_step) * 200

    def size(self) -> int:
        return self._lib.isx_pool_size(self._p)

    def GetRealCols(self) -> int:
        return self._lib.isx_pool_real_cols(self._p)

    def ComputeBatch(self, pairwise: bool, disparity: np.ndarray, segmentation: np.ndarray, roads: Sequence[dict],
                     sections_out: Optional[np.ndarray] = None):
        n = len(roads)
        disparity = np.ascontiguousarray(disparity, dtype=np.float32)
        segmentation = np.ascontiguousarray(segmentation, dtype=np.int32)
        if sections_out is None:
            sections_out = np.zeros((n, self.GetRealCols(), 200), dtype=L.SECTION_DTYPE)
        inst = np.empty(self._inst_cap * n, dtype=L.INSTANCE_DTYPE)
        offs = np.zeros(n + 1, dtype=np.int32)
        rc = self._lib.isx_pool_compute_host(self._p, int(pairwise), n, disparity.ctypes.data,
                                             segmentation.ctypes.data, _roads(roads), sections_out.ctypes.data,
                                             inst.ctypes.data, inst.size, offs.ctypes.data)
        if rc != L.ISX_OK:
            raise StixelsError(f"isx_pool_compute_host: {self._lib.isx_pool_last_error(self._p).decode()} ({rc})")
        return sections_out, inst[:offs[n]].copy(), offs

    def frames_by_worker(self):
        """Frames every worker processed in the last ComputeBatch (its block, less or plus what was taken over)."""
        n = self.size()
        buf = (C.c_int * n)()
        k = self._lib.isx_pool_frames_by_worker(self._p, buf, n)
        return [int(buf[i]) for i in range(k)]

    def close(self):
        if self._p:
            self._lib.isx_pool_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def make_stixels(preset: dict, max_batch: int = 1, device: int = 0) -> Stixels:
    """SetConfig + Initialize from a synth.preset() dict."""
    s = Stixels(device)
    s.SetConfig(StixelConfig(**preset))
    s.Initialize(max_batch)
    return s
