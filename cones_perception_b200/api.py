"""ctypes binding of libconesgpu.so (include/conesgpu.h).

``ConesGpu`` is a thin owner of one ``cp_handle``.  Nothing here computes on the CPU: if the
library is missing or no B200 is present the constructor raises — there is no fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .params import CDetectParams, CGroundParams, DetectParams, GroundParams, to_c_detect, to_c_ground
from .pointcloud2 import CCloudView, PointCloud2, make_view

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libconesgpu.so")

CP_OK, CP_E_PARAM, CP_E_BADFIELD, CP_E_CAPACITY, CP_E_CUDA, CP_E_NOMEM, CP_E_STATE = range(7)

TAP_SECTOR_LOW, TAP_CROP_INDEX, TAP_CROP_POINTS, TAP_CROP_OFFSETS, TAP_VOXEL_KEYS, TAP_VOXEL_ORDER, \
    TAP_VOXEL_CLOUD, TAP_VOXEL_OFFSETS, TAP_LABELS, TAP_PLANE_HYPOTHESES, TAP_PLANE_COUNTS = range(11)

# every symbol include/conesgpu.h declares
ABI_SYMBOLS = [
    "cp_strerror", "cp_last_error", "cp_abi_version", "cp_create_error", "cp_create", "cp_destroy",
    "cp_ground_remove", "cp_detect", "cp_batch_set_device_input", "cp_batch_set_host_input", "cp_batch_run",
    "cp_sync", "cp_batch_results", "cp_detect_batch", "cp_last_run_ms", "cp_last_launch_count", "cp_stream",
    "cp_debug_tap", "cp_debug_sort", "cp_set_stage_timing", "cp_stage_ms", "cp_debug_timeline", "cp_debug_atan2f", "cp_device_results",
    "cp_gather_create", "cp_gather_open", "cp_gather_seq", "cp_gather_wait", "cp_gather_read",
    "cp_last_rows_loaded", "cp_last_pairs", "cp_cone_crops", "cp_cone_images", "cp_rasterize_crops",
    "cp_pinned_alloc", "cp_pinned_free",
    "cp_color_net_load", "cp_color_net_load_tflite", "cp_cone_colors", "cp_classify_images",
    "cp_batch_cone_colors", "cp_batch_track", "cp_track_reset", "cp_debug_track",
    "cp_batch_ground_remove", "cp_batch_ground_device_output", "cp_set_color_cloud",
    "cp_set_ground_plane", "cp_ground_planes",
]

CONE_IMG_ROWS, CONE_IMG_COLS = 15, 12
CONE_EMPTY, CONE_BAD_INDEX, CONE_BAD_INTENSITY, CONE_AMBIGUOUS, CONE_LOW_CONFIDENCE = 1, 2, 4, 8, 16
COLOR_CLOUD_STAGED, COLOR_CLOUD_GROUNDLESS = 0, 1   # cp_set_color_cloud
COLOR_NO_ANSWER = 255   # cp_cone_colors: the service would skip this cone (empty crop) or raise (bad crop)

CLUSTER_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("size", np.uint32), ("min_index", np.uint32)])
TRACKED_CONE_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("cluster", np.uint32), ("color", np.uint32)])
COUNTER_DTYPE = np.dtype([(n, np.uint32) for n in (
    "n_points", "n_ground_kept", "n_cropped", "n_voxels", "n_components", "n_clusters", "key_bits", "passthrough")])


class CConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_points", C.c_uint64), ("max_frames", C.c_uint32),
                ("max_point_step", C.c_uint32), ("max_survivors", C.c_uint64), ("max_voxels", C.c_uint64)]


class CColorNet(C.Structure):
    """cp_color_net."""
    _fields_ = [("c1", C.c_uint32), ("c2", C.c_uint32), ("n_classes", C.c_uint32)] + \
               [(n, C.c_void_p) for n in ("conv1_w", "conv1_b", "conv2_w", "conv2_b", "bn_scale", "bn_shift",
                                          "dense_w", "dense_b")] + [("threshold", C.c_float)]


class CTrackParams(C.Structure):
    """cp_track_params: the ConeDetector members that decide what is published (src/cone_detection.cpp:276-340)."""
    _fields_ = [("classify_colors", C.c_int32), ("use_points_buffer", C.c_int32),
                ("cones_matching_dist_theshold", C.c_double), ("cone_position_extension_length", C.c_double),
                ("cone_width", C.c_float)]


def track_params(classify_colors=False, use_points_buffer=False, match=0.5, ext=0.05, cone_width=0.228):
    return CTrackParams(int(classify_colors), int(use_points_buffer), match, ext, cone_width)


class CTrackedCone(C.Structure):
    """cp_tracked_cone."""
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("cluster", C.c_uint32), ("color", C.c_uint32)]


class CPlaneParams(C.Structure):
    """cp_plane_params: the plane ground model (cp_set_ground_plane).  PARITY UNPINNED: the reference has none."""
    _fields_ = [("seed", C.c_uint64), ("n_hypotheses", C.c_uint32), ("inlier_distance", C.c_float),
                ("ground_height", C.c_float), ("max_tilt_deg", C.c_float)]


def plane_params(seed=0, n_hypotheses=64, inlier_distance=0.1, ground_height=0.1, max_tilt_deg=15.0) -> CPlaneParams:
    """cp_plane_params from keywords (anything with these attribute names also works with set_ground_plane)."""
    return CPlaneParams(int(seed), int(n_hypotheses), float(inlier_distance), float(ground_height), float(max_tilt_deg))


class ConesGpuError(RuntimeError):
    def __init__(self, status: int, detail: str):
        super().__init__(f"libconesgpu status {status}: {detail}")
        self.status = status
        self.detail = detail


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """Load libconesgpu.so and declare the prototypes.  Fails loudly when it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("CONESGPU_LIB") or LIB_PATH   # CONESGPU_LIB: an instrumented build, for debugging
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} is missing: build it with `python -m cones_perception_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(p)
    vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
    lib.cp_strerror.restype = C.c_char_p
    lib.cp_strerror.argtypes = [C.c_int]
    lib.cp_last_error.restype = C.c_char_p
    lib.cp_last_error.argtypes = [vp]
    lib.cp_create_error.restype = C.c_char_p
    lib.cp_abi_version.restype = u32
    lib.cp_create.argtypes = [C.POINTER(vp), C.POINTER(CConfig)]
    lib.cp_destroy.argtypes = [vp]
    lib.cp_destroy.restype = None
    lib.cp_ground_remove.argtypes = [vp, C.POINTER(CCloudView), C.POINTER(CGroundParams), vp, C.POINTER(u32), vp]
    lib.cp_detect.argtypes = [vp, C.POINTER(CCloudView), C.POINTER(CDetectParams), C.POINTER(CGroundParams), vp, u32,
                              C.POINTER(u32), vp]
    lib.cp_batch_set_device_input.argtypes = [vp, vp, u32, vp, u32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    lib.cp_batch_set_host_input.argtypes = [vp, C.POINTER(CCloudView), u32]
    lib.cp_batch_run.argtypes = [vp, C.POINTER(CDetectParams), C.POINTER(CGroundParams)]
    lib.cp_sync.argtypes = [vp]
    lib.cp_batch_results.argtypes = [vp, vp, vp, vp, u64, C.POINTER(u64)]
    lib.cp_detect_batch.argtypes = [vp, C.POINTER(CCloudView), u32, C.POINTER(CDetectParams),
                                    C.POINTER(CGroundParams), vp, vp, vp, u64, C.POINTER(u64)]
    lib.cp_last_run_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.cp_last_launch_count.argtypes = [vp]
    lib.cp_last_launch_count.restype = u32
    lib.cp_stream.argtypes = [vp]
    lib.cp_stream.restype = vp
    lib.cp_debug_tap.argtypes = [vp, C.c_int, vp, u64, C.POINTER(u64)]
    lib.cp_debug_sort.argtypes = [vp, vp, vp, u32, u32]
    lib.cp_set_stage_timing.argtypes = [vp, C.c_int]
    lib.cp_stage_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    lib.cp_debug_timeline.argtypes = [vp, vp, vp]
    lib.cp_debug_atan2f.argtypes = [vp, vp, vp, u32, vp]
    lib.cp_device_results.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.cp_gather_create.argtypes = [vp, u32, u32, vp]
    lib.cp_gather_open.argtypes = [vp, vp, u32, u32, u32]
    lib.cp_gather_seq.argtypes = [vp]
    lib.cp_gather_seq.restype = u32
    lib.cp_gather_wait.argtypes = [vp, u32, u32]
    lib.cp_gather_read.argtypes = [vp, u32, vp, u64]
    lib.cp_last_rows_loaded.argtypes = [vp]
    lib.cp_last_rows_loaded.restype = u64
    lib.cp_last_pairs.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    lib.cp_last_pairs.restype = None
    lib.cp_cone_crops.argtypes = [vp, C.POINTER(CCloudView), u32, vp, u32, C.c_float, vp, vp, u32]
    lib.cp_cone_images.argtypes = [vp, C.POINTER(CCloudView), u32, vp, u32, C.c_float, vp, vp, vp]
    lib.cp_rasterize_crops.argtypes = [vp, vp, vp, u32, vp, vp]
    lib.cp_color_net_load.argtypes = [vp, C.POINTER(CColorNet)]
    lib.cp_color_net_load_tflite.argtypes = [vp, vp, C.c_size_t, C.c_float]
    lib.cp_cone_colors.argtypes = [vp, C.POINTER(CCloudView), u32, vp, u32, C.c_float, vp, vp, vp]
    lib.cp_classify_images.argtypes = [vp, vp, u32, vp, vp, vp]
    lib.cp_batch_cone_colors.argtypes = [vp, C.c_float, C.c_double, vp, vp, vp, vp, u64]
    lib.cp_batch_track.argtypes = [vp, C.POINTER(CTrackParams), vp, u32, vp, vp, u64, C.POINTER(u64)]
    lib.cp_track_reset.argtypes = [vp]
    lib.cp_debug_track.argtypes = [vp, C.POINTER(CTrackParams), vp, vp, u32, vp, vp, vp, u32, vp, vp, u64,
                                   C.POINTER(u64)]
    lib.cp_batch_ground_remove.argtypes = [vp, C.POINTER(CGroundParams), vp, u64, vp, vp]
    lib.cp_batch_ground_device_output.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    lib.cp_set_color_cloud.argtypes = [vp, C.c_int32]
    lib.cp_set_ground_plane.argtypes = [vp, C.POINTER(CPlaneParams)]
    lib.cp_ground_planes.argtypes = [vp, vp, vp, vp, u32]
    lib.cp_pinned_alloc.argtypes = [C.c_int32, C.c_size_t, C.c_int32, C.POINTER(vp)]
    lib.cp_pinned_free.argtypes = [vp]
    lib.cp_pinned_free.restype = None
    if path is None:
        _lib = lib
    return lib


class PinnedBuffer:
    """Page-locked host memory from cp_pinned_alloc, exposed as a numpy array (`.array`, uint8) — for message
    buffers the library can DMA from directly.  Allocate it AFTER binding the thread next to the GPU."""

    def __init__(self, nbytes: int, device: int = 0, write_combined: bool = False):
        self.lib = load_library()
        self._p = C.c_void_p()
        st = self.lib.cp_pinned_alloc(device, nbytes, 1 if write_combined else 0, C.byref(self._p))
        if st != CP_OK:
            raise ConesGpuError(st, "cp_pinned_alloc failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self._p.value))

    @property
    def ptr(self) -> int:
        return int(self._p.value)

    def close(self):
        if getattr(self, "_p", None) is not None and self._p.value:
            self.array = None
            self.lib.cp_pinned_free(self._p)
            self._p = C.c_void_p()

    __del__ = close


class ConesGpu:
    """Owner of one cp_handle (one CUDA device, one stream, used by one thread at a time)."""

    def __init__(self, max_points: int, max_frames: int = 1, device: int = 0, max_point_step: int = 16,
                 max_survivors: int = 0, max_voxels: int = 0, taps: bool = False, back_mode: int | None = None,
                 cluster_front: bool | None = None, env: dict | None = None):
        self.lib = load_library()
        self._h = C.c_void_p()
        if taps:
            os.environ["CONESGPU_TAPS"] = "1"
        if back_mode is not None:   # tests: 0..2 shared-memory back half (growing budgets), 3 general path
            os.environ["CONESGPU_BACK_MODE"] = str(back_mode)
        saved_env = {k: os.environ.get(k) for k in (env or {})}   # extra CONESGPU_* switches read by cp_create
        os.environ.update({k: str(v) for k, v in (env or {}).items()})
        prev_cluster = os.environ.get("CONESGPU_CLUSTER_FRONT")
        if cluster_front is not None:   # single-pass 16-CTA-cluster front end on / off
            os.environ["CONESGPU_CLUSTER_FRONT"] = "1" if cluster_front else "0"
        try:
            cfg = CConfig(device, max_points, max_frames, max_point_step, max_survivors, max_voxels)
            st = self.lib.cp_create(C.byref(self._h), C.byref(cfg))
        finally:
            if taps:
                os.environ.pop("CONESGPU_TAPS", None)
            os.environ.pop("CONESGPU_BACK_MODE", None)
            for k, v in saved_env.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
            if cluster_front is not None:
                if prev_cluster is None:
                    os.environ.pop("CONESGPU_CLUSTER_FRONT", None)
                else:
                    os.environ["CONESGPU_CLUSTER_FRONT"] = prev_cluster
        if st != CP_OK:
            raise ConesGpuError(st, self.lib.cp_create_error().decode())
        self.max_points, self.max_frames = max_points, max_frames
        self._keep = None  # keeps batch inputs alive while the device reads them

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.cp_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, st: int):
        if st != CP_OK:
            raise ConesGpuError(st, self.lib.cp_last_error(self._h).decode())

    # ---- node-equivalent calls --------------------------------------------------------
    def ground_remove(self, msg: PointCloud2, g: GroundParams, copy: bool = True):
        """GroundRemover::cloud_handler body (src/ground_removal.cpp:54-79).
        Returns (cloud32 [N,8] float32 in PCL layout, n_kept, low17; low17 None under the plane model)."""
        view = make_view(msg, fake_missing_intensity=False)
        n = msg.n_points
        if getattr(self, "_gr_n", None) != n:            # the output buffer is reused between calls (a node
            self._gr_out = np.empty((n, 8), dtype=np.float32)   # publishes from one message object too)
            self._gr_n = n
        out = self._gr_out
        low = np.empty(17, dtype=np.float32)
        kept = C.c_uint32()
        cg = to_c_ground(g)
        plane = getattr(self, "_plane", False)
        self._ck(self.lib.cp_ground_remove(self._h, C.byref(view), C.byref(cg), out.ctypes.data, C.byref(kept),
                                           None if plane else low.ctypes.data))
        self.n_frames, self.n_points = 1, n   # the frame stays staged
        return out.copy() if copy else out, kept.value, None if plane else low

    def detect(self, msg: PointCloud2, d: DetectParams, g: GroundParams | None = None, cap: int = 4096,
               fake_missing_intensity: bool = True):
        """ConeDetector::cloud_handler hot path (src/cone_detection.cpp:151-167 + :261-273).
        Returns (clusters structured array, counters structured scalar)."""
        view = make_view(msg, fake_missing_intensity)
        if getattr(self, "_det_cap", None) != cap:       # output buffers are reused between calls
            self._det_out = np.zeros(cap, dtype=CLUSTER_DTYPE)
            self._det_ctr = np.zeros(1, dtype=COUNTER_DTYPE)
            self._det_cap = cap
        out, ctr = self._det_out, self._det_ctr
        k = C.c_uint32()
        cd = to_c_detect(d)
        cg = to_c_ground(g) if g is not None else None
        self._ck(self.lib.cp_detect(self._h, C.byref(view), C.byref(cd), C.byref(cg) if cg is not None else None,
                                    out.ctypes.data, cap, C.byref(k), ctr.ctypes.data))
        self.n_frames, self.n_points = 1, msg.n_points   # the run is one frame (results(), batch_track())
        return out[:k.value].copy(), ctr[0].copy()

    # ---- colour path inputs (SURVEY §8 f3) ----------------------------------------------
    @staticmethod
    def _centers(centers) -> np.ndarray:
        return np.ascontiguousarray(np.asarray(centers, dtype=np.float32).reshape(-1, 2))

    def cone_crops(self, centers, cone_width: float = 0.228, msg: PointCloud2 | None = None, frame: int = 0,
                   cap_points: int = 1 << 16, fake_missing_intensity: bool = True):
        """get_reconstructed_cone (src/cone_detection.cpp:222-238) for all centres at once.  msg=None
        reuses frame `frame` of the input already staged on the device.  Returns (offsets, xyzi)."""
        c = self._centers(centers)
        view = make_view(msg, fake_missing_intensity) if msg is not None else None
        off = np.zeros(len(c) + 1, np.uint32)
        pts = np.empty((cap_points, 4), np.float32)
        self._ck(self.lib.cp_cone_crops(self._h, C.byref(view) if view is not None else None, frame, c.ctypes.data,
                                        len(c), cone_width, off.ctypes.data, pts.ctypes.data, cap_points))
        return off, pts[:off[-1]].copy()

    def cone_images(self, centers, cone_width: float = 0.228, msg: PointCloud2 | None = None, frame: int = 0,
                    fake_missing_intensity: bool = True):
        """Crops + ColorClassifier.to_image (scripts/color_classifier_server.py:130-156) on the device.
        Returns (images [n,15,12] uint8, counts, flags)."""
        c = self._centers(centers)
        view = make_view(msg, fake_missing_intensity) if msg is not None else None
        img = np.zeros((len(c), CONE_IMG_ROWS, CONE_IMG_COLS), np.uint8)
        counts, flags = np.zeros(len(c), np.uint32), np.zeros(len(c), np.uint32)
        self._ck(self.lib.cp_cone_images(self._h, C.byref(view) if view is not None else None, frame, c.ctypes.data,
                                         len(c), cone_width, img.ctypes.data, counts.ctypes.data, flags.ctypes.data))
        return img, counts, flags

    def rasterize_crops(self, xyzi: np.ndarray, offsets):
        """to_image on host crops (packed x,y,z,intensity rows + offsets).  Returns (images, flags)."""
        a = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
        off = np.ascontiguousarray(offsets, np.uint32)
        n = len(off) - 1
        img = np.zeros((n, CONE_IMG_ROWS, CONE_IMG_COLS), np.uint8)
        flags = np.zeros(n, np.uint32)
        self._ck(self.lib.cp_rasterize_crops(self._h, a.ctypes.data, off.ctypes.data, n, img.ctypes.data,
                                             flags.ctypes.data))
        return img, flags

    # ---- colour classifier (models/dam_net) ---------------------------------------------
    def color_net_load_tflite(self, model, threshold: float = 0.8):
        """Load the reference's classifier from a .tflite file (path or bytes): what
        scripts/color_classifier_server.py:66 hands to tf.lite.Interpreter."""
        data = model if isinstance(model, (bytes, bytearray)) else open(model, "rb").read()
        buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
        self._ck(self.lib.cp_color_net_load_tflite(self._h, buf, len(data), threshold))
        self._n_classes = None

    def color_net_load(self, conv1_w, conv1_b, conv2_w, conv2_b, bn_scale, bn_shift, dense_w, dense_b,
                       threshold: float = 0.8):
        """Raw tensors in the flatbuffer's layouts: conv [out][3][3][in], dense [classes][2*c2]."""
        t = [np.ascontiguousarray(a, np.float32) for a in (conv1_w, conv1_b, conv2_w, conv2_b, bn_scale, bn_shift,
                                                           dense_w, dense_b)]
        net = CColorNet(t[0].shape[0], t[2].shape[0], t[6].shape[0], *[a.ctypes.data for a in t], threshold)
        self._ck(self.lib.cp_color_net_load(self._h, C.byref(net)))
        self._n_classes = t[6].shape[0]

    def classify_images(self, images: np.ndarray, n_classes: int = 3):
        """The network alone on [n,15,12] uint8 images.  Returns (colors u8 [n], probs [n,classes], logits)."""
        img = np.ascontiguousarray(images, np.uint8).reshape(-1, CONE_IMG_ROWS, CONE_IMG_COLS)
        n = len(img)
        nc = getattr(self, "_n_classes", None) or n_classes
        colors = np.zeros(n, np.uint8)
        probs, logits = np.zeros((n, nc), np.float32), np.zeros((n, nc), np.float32)
        self._ck(self.lib.cp_classify_images(self._h, img.ctypes.data, n, colors.ctypes.data, probs.ctypes.data,
                                             logits.ctypes.data))
        return colors, probs, logits

    def cone_colors(self, centers, cone_width: float = 0.228, msg: PointCloud2 | None = None, frame: int = 0,
                    fake_missing_intensity: bool = True, n_classes: int = 3):
        """handle_classify_color (scripts/color_classifier_server.py:78-126) on the device for all centres:
        box gather -> to_image -> network.  Returns (colors u8 [n] with 255 = no answer, probs, flags)."""
        c = self._centers(centers)
        view = make_view(msg, fake_missing_intensity) if msg is not None else None
        nc = getattr(self, "_n_classes", None) or n_classes
        colors = np.zeros(len(c), np.uint8)
        probs, flags = np.zeros((len(c), nc), np.float32), np.zeros(len(c), np.uint32)
        self._ck(self.lib.cp_cone_colors(self._h, C.byref(view) if view is not None else None, frame, c.ctypes.data,
                                         len(c), cone_width, colors.ctypes.data, probs.ctypes.data, flags.ctypes.data))
        return colors, probs, flags

    def batch_cone_colors(self, cone_width: float = 0.228, extension_length: float = 0.05, n_classes: int = 3):
        """handle_classify_color for every cluster record of the last run, at its centroid extended by
        extension_length (src/cone_detection.cpp:276-278), on the run's own input.  Returns (colors u8 [K] with
        255 = no answer, probs [K, classes], flags u32 [K], counts u32 [K] crop points), aligned with results()."""
        total = C.c_uint64()
        self._ck(self.lib.cp_batch_results(self._h, None, None, None, 0, C.byref(total)))
        K = total.value
        nc = getattr(self, "_n_classes", None) or n_classes
        colors, probs = np.zeros(K, np.uint8), np.zeros((K, nc), np.float32)
        flags, counts = np.zeros(K, np.uint32), np.zeros(K, np.uint32)
        self._ck(self.lib.cp_batch_cone_colors(self._h, cone_width, extension_length, colors.ctypes.data,
                                               probs.ctypes.data, flags.ctypes.data, counts.ctypes.data, K))
        return colors, probs, flags, counts

    def set_color_cloud(self, groundless: bool):
        """Crop colours of the staged input (cone_* with msg=None, batch_cone_colors, batch_track in colour mode) from
        the ground node's message of each frame after a run with ground removal (groundless=True), as the reference's
        two-node launch does, or from the staged cloud itself (False, the default)."""
        self._ck(self.lib.cp_set_color_cloud(self._h, COLOR_CLOUD_GROUNDLESS if groundless else COLOR_CLOUD_STAGED))

    # ---- what the node publishes, over frame sequences ----------------------------------
    @staticmethod
    def _seqs(seq_offsets):
        if seq_offsets is None:
            return None, 1
        so = np.ascontiguousarray(seq_offsets, np.uint32)
        return so, len(so) - 1

    def batch_track(self, params: CTrackParams, seq_offsets=None):
        """The radial extension, temporal gate / points buffer, colour carry-over and response rules of the
        cone-detection node (src/cone_detection.cpp:276-340) for every frame of the last run; sequence s continues
        state slot s.  Returns (cones TRACKED_CONE_DTYPE [n], cloud_offsets u32 [4F + 1]): cloud c of frame f is
        cones[cloud_offsets[4f + c]:cloud_offsets[4f + c + 1]]."""
        total = C.c_uint64()
        self._ck(self.lib.cp_batch_results(self._h, None, None, None, 0, C.byref(total)))
        so, n_seqs = self._seqs(seq_offsets)
        out = np.zeros(total.value, TRACKED_CONE_DTYPE)
        coff = np.zeros(4 * self.n_frames + 1, np.uint32)
        n = C.c_uint64()
        self._ck(self.lib.cp_batch_track(self._h, C.byref(params), so.ctypes.data if so is not None else None, n_seqs,
                                         out.ctypes.data, coff.ctypes.data, len(out), C.byref(n)))
        return out[:n.value].copy(), coff

    def track_reset(self):
        """Clears every state slot: each behaves like a node that has just started."""
        self._ck(self.lib.cp_track_reset(self._h))

    def debug_track(self, params: CTrackParams, records, record_offsets, colors=None, flags=None, seq_offsets=None):
        """cp_batch_track's kernels on caller-supplied records (CLUSTER_DTYPE) and per-record service answers."""
        rec = np.ascontiguousarray(records, CLUSTER_DTYPE)
        roff = np.ascontiguousarray(record_offsets, np.uint32)
        F = len(roff) - 1
        col = np.ascontiguousarray(colors if colors is not None else np.zeros(len(rec)), np.uint8)
        fl = np.ascontiguousarray(flags if flags is not None else np.zeros(len(rec)), np.uint32)
        so, n_seqs = self._seqs(seq_offsets)
        out = np.zeros(len(rec), TRACKED_CONE_DTYPE)
        coff = np.zeros(4 * F + 1, np.uint32)
        n = C.c_uint64()
        self._ck(self.lib.cp_debug_track(self._h, C.byref(params), rec.ctypes.data, roff.ctypes.data, F,
                                         col.ctypes.data, fl.ctypes.data, so.ctypes.data if so is not None else None,
                                         n_seqs, out.ctypes.data, coff.ctypes.data, len(out), C.byref(n)))
        return out[:n.value].copy(), coff

    # ---- batches ----------------------------------------------------------------------
    def set_device_input(self, d_ptr: int, frame_points, point_step: int = 16, off=(0, 4, 8, 12), keep=None):
        fp = np.ascontiguousarray(frame_points, dtype=np.uint32)
        self._keep = keep
        self._ck(self.lib.cp_batch_set_device_input(self._h, C.c_void_p(d_ptr), len(fp), fp.ctypes.data, point_step,
                                                    off[0], off[1], off[2], off[3]))
        self.n_frames = len(fp)
        self.n_points = int(fp.sum(dtype=np.uint64))

    def set_host_input(self, msgs, fake_missing_intensity: bool = True):
        views = (CCloudView * len(msgs))(*[make_view(m, fake_missing_intensity) for m in msgs])
        self._keep = msgs
        self._ck(self.lib.cp_batch_set_host_input(self._h, views, len(msgs)))
        self.n_frames = len(msgs)
        self.n_points = sum(m.n_points for m in msgs)

    def batch_ground_remove(self, g: GroundParams, host: bool = True):
        """GroundRemover::cloud_handler (src/ground_removal.cpp:54-79) for every frame of the staged batch (stage host
        clouds with fake_missing_intensity=False, as the ground node reads them).  Returns (cloud32 [sum N_f, 8]
        float32, frame f's message at rows P_f .. P_f + N_f, or None when host is False; n_kept u32 [F];
        low f32 [F, 17], None under the plane model).  The messages stay on the device: ground_device_output()."""
        plane = getattr(self, "_plane", False)
        out = np.empty((self.n_points, 8), np.float32) if host else None
        kept = np.zeros(self.n_frames, np.uint32)
        low = np.zeros((self.n_frames, 17), np.float32)
        cg = to_c_ground(g)
        self._ck(self.lib.cp_batch_ground_remove(self._h, C.byref(cg), out.ctypes.data if host else None,
                                                 self.n_points if host else 0, kept.ctypes.data,
                                                 None if plane else low.ctypes.data))
        return out, kept, None if plane else low

    def ground_device_output(self):
        """(device pointer, n_points) of the messages of the last batch_ground_remove (32 B per point)."""
        p, n = C.c_void_p(), C.c_uint64()
        self._ck(self.lib.cp_batch_ground_device_output(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def set_ground_plane(self, p=None):
        """The plane ground model (cp_set_ground_plane) for every later call with ground params, or the sector model
        (the default) with p None.  p: a CPlaneParams or anything with its field names (oracle.plane_oracle.PlaneParams)."""
        if p is None:
            self._ck(self.lib.cp_set_ground_plane(self._h, None))
            self._plane = False
            return
        c = p if isinstance(p, CPlaneParams) else plane_params(p.seed, p.n_hypotheses, p.inlier_distance,
                                                                 p.ground_height, p.max_tilt_deg)
        self._ck(self.lib.cp_set_ground_plane(self._h, C.byref(c)))
        self._plane = True

    def ground_planes(self):
        """The plane each frame chose in the last run or ground call with the plane model: (planes f32 [F, 4] a, b, c, d,
        inliers u32 [F], hypothesis i32 [F], -1 where no hypothesis was valid)."""
        F = self.n_frames
        planes = np.zeros((F, 4), np.float32)
        inl = np.zeros(F, np.uint32)
        hyp = np.zeros(F, np.int32)
        self._ck(self.lib.cp_ground_planes(self._h, planes.ctypes.data, inl.ctypes.data, hyp.ctypes.data, F))
        return planes, inl, hyp

    def run(self, d: DetectParams, g: GroundParams | None = None):
        cd = to_c_detect(d)
        cg = to_c_ground(g) if g is not None else None
        self._ck(self.lib.cp_batch_run(self._h, C.byref(cd), C.byref(cg) if cg is not None else None))

    def sync(self):
        self._ck(self.lib.cp_sync(self._h))

    def results(self, cap: int | None = None):
        """Returns (counters[F], cluster_offsets[F+1], clusters[K_total])."""
        F = self.n_frames
        ctr = np.zeros(F, dtype=COUNTER_DTYPE)
        off = np.zeros(F + 1, dtype=np.uint32)
        total = C.c_uint64()
        # first call sizes the output
        self._ck(self.lib.cp_batch_results(self._h, ctr.ctypes.data, off.ctypes.data, None, 0, C.byref(total)))
        out = np.zeros(total.value, dtype=CLUSTER_DTYPE)
        if total.value:
            self._ck(self.lib.cp_batch_results(self._h, None, None, out.ctypes.data, total.value, C.byref(total)))
        return ctr, off, out

    def detect_batch(self, msgs, d: DetectParams, g: GroundParams | None = None):
        self.set_host_input(msgs)
        self.run(d, g)
        return self.results()

    def last_run_ms(self) -> float:
        ms = C.c_float()
        self._ck(self.lib.cp_last_run_ms(self._h, C.byref(ms)))
        return ms.value

    def set_stage_timing(self, on: bool):
        self._ck(self.lib.cp_set_stage_timing(self._h, 1 if on else 0))

    def stage_ms(self, stage: int) -> float:
        ms = C.c_float()
        self._ck(self.lib.cp_stage_ms(self._h, stage, C.byref(ms)))
        return ms.value

    def timeline(self, base: "ConesGpu | None" = None) -> np.ndarray:
        """Device timestamps (ms) of the last run relative to the start of `base`'s last run:
        run start, pass 1 start/end, pass 2 start/end, run end (stage timing must be on)."""
        out = np.zeros(6, np.float32)
        self._ck(self.lib.cp_debug_timeline(self._h, base._h if base is not None else None, out.ctypes.data))
        return out

    def debug_atan2f(self, y: np.ndarray, x: np.ndarray) -> np.ndarray:
        y = np.ascontiguousarray(y, np.float32)
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(y)
        self._ck(self.lib.cp_debug_atan2f(self._h, y.ctypes.data, x.ctypes.data, len(y), out.ctypes.data))
        return out

    def device_results(self):
        """(d_clusters, d_cluster_offsets, d_n_clusters) raw device pointers of the last run."""
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._ck(self.lib.cp_device_results(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    # ---- multi-GPU result path over peer memory ------------------------------------------
    def gather_create(self, world: int, slot_words: int) -> bytes:
        """Rank 0: allocate the gather buffer; returns the 64-byte CUDA-IPC handle to broadcast."""
        buf = (C.c_uint8 * 64)()
        self._ck(self.lib.cp_gather_create(self._h, world, slot_words, buf))
        return bytes(buf)

    def gather_open(self, handle: bytes, rank: int, world: int, slot_words: int):
        buf = (C.c_uint8 * 64).from_buffer_copy(handle)
        self._ck(self.lib.cp_gather_open(self._h, buf, rank, world, slot_words))

    def gather_seq(self) -> int:
        return int(self.lib.cp_gather_seq(self._h))

    def gather_wait(self, seq: int, timeout_ms: int = 5000):
        self._ck(self.lib.cp_gather_wait(self._h, seq, timeout_ms))

    def gather_read(self, seq: int, world: int, slot_words: int) -> np.ndarray:
        out = np.empty((world, slot_words), dtype=np.int32)
        self._ck(self.lib.cp_gather_read(self._h, seq, out.ctypes.data, out.nbytes))
        return out

    def last_rows_loaded(self) -> int:
        return int(self.lib.cp_last_rows_loaded(self._h))

    def last_pairs(self) -> tuple[int, int]:
        """(candidate voxel pairs visited, pairs whose distance was tested) by the clustering of the last run."""
        a, b = C.c_uint64(), C.c_uint64()
        self.lib.cp_last_pairs(self._h, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)

    def last_launch_count(self) -> int:
        return int(self.lib.cp_last_launch_count(self._h))

    def stream(self) -> int:
        return int(self.lib.cp_stream(self._h) or 0)

    # ---- parity taps ------------------------------------------------------------------
    def tap(self, which: int) -> np.ndarray:
        dt = {TAP_SECTOR_LOW: np.float32, TAP_CROP_POINTS: np.float32, TAP_VOXEL_CLOUD: np.float32,
              TAP_LABELS: np.int32, TAP_PLANE_HYPOTHESES: np.float32}.get(which, np.uint32)
        width = 4 if which in (TAP_CROP_POINTS, TAP_VOXEL_CLOUD, TAP_PLANE_HYPOTHESES) else 1
        cap = (self.max_points + self.max_frames + 64) * max(1, width) * 4 + self.max_frames * 17 * 4
        if which in (TAP_PLANE_HYPOTHESES, TAP_PLANE_COUNTS):
            cap = self.max_frames * 256 * width * 4
        buf = np.empty(cap // 4, dtype=dt)
        n = C.c_uint64()
        self._ck(self.lib.cp_debug_tap(self._h, which, buf.ctypes.data, buf.nbytes, C.byref(n)))
        out = buf[:n.value * width].copy()
        return out.reshape(-1, 4) if width == 4 else out

    def debug_sort(self, keys: np.ndarray, vals: np.ndarray, bits: int):
        k = np.ascontiguousarray(keys, dtype=np.uint64).copy()
        v = np.ascontiguousarray(vals, dtype=np.uint32).copy()
        self._ck(self.lib.cp_debug_sort(self._h, k.ctypes.data, v.ctypes.data, len(k), bits))
        return k, v
