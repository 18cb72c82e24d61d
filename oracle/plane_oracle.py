"""ctypes wrapper of the plane ground model's CPU restatement (oracle/plane_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED: the reference has no plane model.  detect() is the two-node chain the GPU's fused run must equal:
the plane ground node's message, then the detector without ground removal on it (oracle.detect).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

from . import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "libplaneoracle.so")
SRC = os.path.join(_HERE, "plane_oracle.cpp")

_lib = None


@dataclass
class PlaneParams:
    seed: int = 0
    n_hypotheses: int = 64
    inlier_distance: float = 0.1
    ground_height: float = 0.1
    max_tilt_deg: float = 15.0


def build(force: bool = False) -> str:
    if force or not os.path.exists(LIB) or os.path.getmtime(SRC) > os.path.getmtime(LIB):
        tmp = LIB + f".{os.getpid()}.tmp"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", tmp, SRC], check=True)
        os.replace(tmp, LIB)
    return LIB


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
        L.orc_plane_index.argtypes = [u64, u32, u32, u32]
        L.orc_plane_index.restype = u32
        L.orc_plane_cos_tilt.argtypes = [C.c_float]
        L.orc_plane_cos_tilt.restype = C.c_double
        L.orc_plane_hypotheses.argtypes = [vp, u32, u64, u32, C.c_float, vp]
        L.orc_plane_hypotheses.restype = None
        L.orc_plane_counts.argtypes = [vp, u32, vp, u32, C.c_float, vp]
        L.orc_plane_counts.restype = None
        L.orc_plane_ground_node.argtypes = [vp, u32, u64, u32, C.c_float, C.c_float, C.c_float, vp, C.POINTER(u32), vp,
                                            C.POINTER(u32), C.POINTER(C.c_int32), vp]
        L.orc_plane_ground_node.restype = None
        _lib = L
    return _lib


def _pts(pts: np.ndarray) -> np.ndarray:
    """PointXYZI records (oracle.POINT_DTYPE) from records or a float32 [N, 4] x, y, z, intensity array."""
    if pts.dtype == O.POINT_DTYPE:
        return np.ascontiguousarray(pts)
    return O.points32(pts)


def plane_index(seed: int, h: int, j: int, n: int) -> int:
    return int(lib().orc_plane_index(seed & (2**64 - 1), h, j, n))


def cos_tilt(max_tilt_deg: float) -> float:
    return float(lib().orc_plane_cos_tilt(max_tilt_deg))


def hypotheses(pts: np.ndarray, p: PlaneParams) -> np.ndarray:
    """[H, 4] float32 a, b, c, d per hypothesis (NaN when invalid)."""
    a = _pts(pts)
    out = np.zeros((p.n_hypotheses, 4), np.float32)
    lib().orc_plane_hypotheses(a.ctypes.data, len(a), p.seed, p.n_hypotheses, p.max_tilt_deg, out.ctypes.data)
    return out


def counts(pts: np.ndarray, planes: np.ndarray, inlier_distance: float) -> np.ndarray:
    a = _pts(pts)
    pl = np.ascontiguousarray(planes, np.float32).reshape(-1, 4)
    out = np.zeros(len(pl), np.uint32)
    lib().orc_plane_counts(a.ctypes.data, len(a), pl.ctypes.data, len(pl), inlier_distance, out.ctypes.data)
    return out


def ground_node(pts: np.ndarray, p: PlaneParams):
    """Returns (message [N] PointXYZI records, kept, plane [4], inliers, hypothesis (-1: none), keep mask [N])."""
    a = _pts(pts)
    n = len(a)
    out = np.zeros(n, dtype=O.POINT_DTYPE)
    keep = np.zeros(n, np.uint8)
    plane = np.zeros(4, np.float32)
    kept, inl, hyp = C.c_uint32(), C.c_uint32(), C.c_int32()
    lib().orc_plane_ground_node(a.ctypes.data, n, p.seed, p.n_hypotheses, p.inlier_distance, p.ground_height,
                                p.max_tilt_deg, out.ctypes.data, C.byref(kept), plane.ctypes.data, C.byref(inl),
                                C.byref(hyp), keep.ctypes.data)
    return out, kept.value, plane, inl.value, hyp.value, keep


def view_of_records(rec: np.ndarray) -> O.View:
    """A 32-byte PointXYZI cloud (the ground node's message) as a cloud view."""
    assert rec.dtype == O.POINT_DTYPE and rec.flags["C_CONTIGUOUS"]
    return O.View(rec.ctypes.data, len(rec), 1, 32, 32 * len(rec), 0, 4, 8, 16, 0, 1)


def detect(pts: np.ndarray, p: PlaneParams, d, mode: int = O.CANONICAL):
    """Detect with the plane model: the plane ground node, then the detector without ground removal on its message.
    Returns (clusters, counters with n_ground_kept = G, message, kept)."""
    msg, kept, _, _, _, _ = ground_node(pts, p)
    cl, ctr, _ = O.detect(view_of_records(msg), d, None, mode)
    ctr.n_ground_kept = kept
    return cl, ctr, msg, kept
