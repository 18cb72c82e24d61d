"""CPU tests of the plane ground model's oracle (oracle/plane_oracle.cpp) against an independent numpy / Python
restatement of the contract in include/conesgpu.h (cp_plane_params).  PARITY UNPINNED: the reference has no plane
model; these tests pin the oracle, and tests/test_gpu_plane_ground.py holds the kernels to the oracle."""
import math

import numpy as np
import pytest

from cones_perception_b200 import scans
from cones_perception_b200.params import PRESETS, GroundParams
from oracle import oracle as O
from oracle import plane_oracle as PO

M64 = (1 << 64) - 1


def splitmix64(x):
    z = (x + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def draw(seed, h, j, n):
    return ((splitmix64((seed + 3 * h + j) & M64) >> 32) * n) >> 32


def plane_py(p0, p1, p2, cos_t):
    """The contract's plane in Python floats (IEEE double, every operation rounded on its own)."""
    P = [tuple(float(v) for v in p[:3]) for p in (p0, p1, p2)]
    if not all(math.isfinite(v) for p in P for v in p):
        return None
    (x0, y0, z0), (x1, y1, z1), (x2, y2, z2) = P
    ux, uy, uz = x1 - x0, y1 - y0, z1 - z0
    vx, vy, vz = x2 - x0, y2 - y0, z2 - z0
    nx, ny, nz = uy * vz - uz * vy, uz * vx - ux * vz, ux * vy - uy * vx
    L = math.sqrt(nx * nx + ny * ny + nz * nz)
    if not (L > 0.0) or not math.isfinite(L):
        return None
    if nz < 0.0:
        nx, ny, nz = -nx, -ny, -nz
    if nz / L < cos_t:
        return None
    nx, ny, nz = nx / L, ny / L, nz / L
    d = -(nx * x0 + ny * y0 + nz * z0)
    return np.array([nx, ny, nz, d], np.float32)


def hypotheses_py(xyz, p):
    n = len(xyz)
    cos_t = math.cos(float(np.float32(p.max_tilt_deg)) * (math.pi / 180.0))
    out = np.full((p.n_hypotheses, 4), np.nan, np.float32)
    if n < 3:
        return out
    for h in range(p.n_hypotheses):
        pl = plane_py(*(xyz[draw(p.seed, h, j, n)] for j in range(3)), cos_t)
        if pl is not None:
            out[h] = pl
    return out


def scan(cfg_id=2, seed=0):
    cfg = scans.config(cfg_id)
    return cfg, np.ascontiguousarray(scans.generate(cfg, 1, seed)[0])


def rotate(p, pitch_deg, roll_deg):
    a, b = np.radians(pitch_deg), np.radians(roll_deg)
    Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    Rx = np.array([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]])
    R = Rx @ Ry
    q = p.astype(np.float64)
    q[:, :3] = q[:, :3] @ R.T
    return np.ascontiguousarray(q.astype(np.float32)), R


def test_splitmix_indices():
    rng = np.random.default_rng(1)
    for _ in range(300):
        seed = int(rng.integers(0, 2**63)) * 2 + int(rng.integers(0, 2))
        h, j = int(rng.integers(0, 256)), int(rng.integers(0, 3))
        n = int(rng.choice([1, 3, 7, 2049, 131072, 2**31 - 1]))
        got = PO.plane_index(seed, h, j, n)
        assert got == draw(seed, h, j, n) and got < n
    assert PO.plane_index(M64, 255, 2, 1000) == draw(M64, 255, 2, 1000)   # seed + 3h + j wraps modulo 2^64


@pytest.mark.parametrize("pitch,roll", [(0, 0), (2, 0), (0, 4), (3, -3)])
def test_plane_coefficients_bit_exact(pitch, roll):
    _, base = scan()
    pts, _ = rotate(base, pitch, roll)
    p = PO.PlaneParams(seed=7, n_hypotheses=64)
    got = PO.hypotheses(pts, p)
    exp = hypotheses_py(pts[:, :3], p)
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))
    assert np.isfinite(got[:, 0]).sum() > 10


def test_inlier_counts_outside_guard_band():
    _, base = scan()
    pts, _ = rotate(base, 2, 1)
    p = PO.PlaneParams(seed=3, n_hypotheses=32, inlier_distance=0.1)
    planes = PO.hypotheses(pts, p)
    x, y, z = (pts[:, i].astype(np.float64) for i in range(3))
    checked = 0
    for h, pl in enumerate(planes):
        if np.isnan(pl[0]):
            continue
        s = pl[0].astype(np.float64) * x + pl[1] * y + pl[2] * z + pl[3]
        far = np.abs(np.abs(s) - 0.1) > 1e-6
        got = PO.counts(pts[far], pl[None], 0.1)[0]
        assert got == int((np.abs(s[far]) <= 0.1).sum())
        checked += 1
    assert checked > 5


def test_known_answers():
    rng = np.random.default_rng(0)
    n = 500
    flat = np.zeros((n, 4), np.float32)
    flat[:, 0] = rng.uniform(-10, 10, n)
    flat[:, 1] = rng.uniform(-10, 10, n)
    flat[:, 2] = -0.6
    msg, kept, plane, inl, hyp, keep = PO.ground_node(flat, PO.PlaneParams(n_hypotheses=16))
    assert hyp >= 0 and inl == n and kept == 0 and not keep.any()
    assert plane[0] == 0 and plane[1] == 0 and plane[2] == 1 and plane[3] == np.float32(0.6)
    # a tilted plane z = 0.1 x - 0.05 y - 0.5 is recovered
    t = np.zeros((n, 4), np.float32)
    t[:, 0] = rng.uniform(-10, 10, n)
    t[:, 1] = rng.uniform(-10, 10, n)
    t[:, 2] = 0.1 * t[:, 0].astype(np.float64) - 0.05 * t[:, 1] - 0.5
    _, _, plane, inl, hyp, _ = PO.ground_node(t, PO.PlaneParams(n_hypotheses=16, inlier_distance=0.01))
    exp = np.array([-0.1, 0.05, 1.0, 0.5]) / math.sqrt(1 + 0.01 + 0.0025)
    assert hyp >= 0 and inl == n and np.allclose(plane, exp, atol=1e-5)


def test_degenerate_triples():
    ct = math.cos(math.radians(15.0))
    p = np.array([1.0, 2.0, -0.6, 0], np.float32)
    q = np.array([3.0, 1.0, -0.6, 0], np.float32)
    assert plane_py(p, p, q, ct) is None                                  # repeated point: n = 0
    assert plane_py(p, q, 2 * q - p, ct) is None                          # collinear
    assert plane_py(p, q, np.array([np.nan, 0, 0, 0], np.float32), ct) is None
    # the oracle agrees: a 3-point frame whose draws repeat an index, a collinear frame, a NaN sample
    pp = PO.PlaneParams(seed=0, n_hypotheses=256)
    tri = np.stack([p, q, np.array([2.0, 5.0, -0.6, 0], np.float32)])
    planes = PO.hypotheses(tri, pp)
    for h in range(256):
        ids = {draw(0, h, j, 3) for j in range(3)}
        assert np.isnan(planes[h, 0]) == (len(ids) < 3)
    col = np.stack([p, q, 2 * q - p, 3 * q - 2 * p]).astype(np.float32)
    assert np.isnan(PO.hypotheses(col, pp)[:, 0]).all()
    nan_pt = tri.copy()
    nan_pt[1, 2] = np.nan
    got = PO.hypotheses(nan_pt, pp)
    for h in range(256):
        ids = [draw(0, h, j, 3) for j in range(3)]
        if 1 in ids:
            assert np.isnan(got[h, 0])
    _, kept, _, _, _, keep = PO.ground_node(nan_pt, pp)
    assert keep[1] == 0   # a non-finite point is always dropped


def test_tilt_gate_rejects_a_wall():
    rng = np.random.default_rng(2)
    n = 300
    wall = np.zeros((n, 4), np.float32)
    wall[:, 0] = 5.0
    wall[:, 1] = rng.uniform(-3, 3, n)
    wall[:, 2] = rng.uniform(-0.5, 2, n)
    _, kept, plane, inl, hyp, keep = PO.ground_node(wall, PO.PlaneParams(n_hypotheses=64))
    assert hyp == -1 and inl == 0 and np.isnan(plane).all() and kept == n and keep.all()
    assert np.isnan(PO.hypotheses(wall, PO.PlaneParams(n_hypotheses=64))[:, 0]).all()


def test_ties_go_to_the_lowest_hypothesis():
    rng = np.random.default_rng(3)
    n = 64
    flat = np.zeros((n, 4), np.float32)
    flat[:, 0] = rng.uniform(-10, 10, n)
    flat[:, 1] = rng.uniform(-10, 10, n)
    flat[:, 2] = -0.6
    p = PO.PlaneParams(seed=11, n_hypotheses=32)
    planes = PO.hypotheses(flat, p)
    cnt = PO.counts(flat, planes, p.inlier_distance)
    valid = ~np.isnan(planes[:, 0])
    assert (cnt[valid] == n).all() and valid.sum() > 1   # every valid hypothesis ties
    _, _, _, _, hyp, _ = PO.ground_node(flat, p)
    assert hyp == int(np.flatnonzero(valid)[0])


@pytest.mark.parametrize("n", [0, 1, 2, 3])
def test_tiny_frames(n):
    pts = np.array([[1, 0, -0.6, 5], [0, 1, -0.6, 6], [2, 3, -0.5, 7]], np.float32)[:n].copy()
    p = PO.PlaneParams(n_hypotheses=8)
    planes = PO.hypotheses(pts, p)
    assert np.array_equal(planes.view(np.uint32), hypotheses_py(pts[:, :3], p).view(np.uint32))
    msg, kept, plane, inl, hyp, keep = PO.ground_node(pts, p)
    if n < 3:
        assert np.isnan(planes).all() and hyp == -1 and kept == n and keep.all()
    assert len(msg) == n
    assert np.array_equal(msg["x"][:kept], pts[keep.astype(bool), 0])
    assert (msg["pad"] == 1.0).all() and (msg["x"][kept:] == 0).all()


def test_message_matches_restated_verdict():
    _, base = scan()
    pts, _ = rotate(base, 2, 0)
    pts[::997, 2] = np.nan
    p = PO.PlaneParams(seed=5)
    msg, kept, plane, inl, hyp, keep = PO.ground_node(pts, p)
    planes = PO.hypotheses(pts, p)
    cnt = PO.counts(pts, planes, p.inlier_distance)
    valid = ~np.isnan(planes[:, 0])
    best = max(np.flatnonzero(valid), key=lambda h: (cnt[h], -h))
    assert hyp == best and inl == cnt[best] and np.array_equal(plane.view(np.uint32), planes[best].view(np.uint32))
    x, y, z = (pts[:, i].astype(np.float64) for i in range(3))
    s = plane[0].astype(np.float64) * x + plane[1] * y + plane[2] * z + plane[3]
    far = np.abs(s - p.ground_height) > 1e-6
    fin = np.isfinite(pts[:, :3]).all(1)
    assert np.array_equal(keep.astype(bool)[far], (fin & (s >= p.ground_height))[far])
    assert kept == keep.sum()
    assert np.array_equal(msg["z"][:kept], pts[keep.astype(bool), 2]) and (msg["z"][kept:] == 0).all()


def _on_cone(cl, cones_xy):
    if len(cl) == 0:
        return 0
    xy = np.c_[cl["x"], cl["y"]]
    return int(sum(np.min(np.hypot(*(cones_xy - k).T)) < 0.3 for k in xy))


def test_pitched_and_rolled_scans_keep_their_cones():
    cfg, base = scan()
    d, g = PRESETS["simulation"], GroundParams()
    p = PO.PlaneParams(seed=0, n_hypotheses=64)
    hits = {}
    for pitch, roll in [(0, 0), (2, 0), (0, 4)]:
        pts, R = rotate(base, pitch, roll)
        cw = (np.c_[cfg.cones, np.full(len(cfg.cones), -cfg.sensor_h + 0.16)] @ R.T)[:, :2]
        cl_plane, ctr, _, _ = PO.detect(pts, p, d)
        cl_sector, _, _ = O.detect(O.view_of_xyzi(pts), d, g)
        hits[(pitch, roll)] = (_on_cone(cl_plane, cw), _on_cone(cl_sector, cw))
    level_plane, level_sector = hits[(0, 0)]
    assert level_plane >= level_sector > 0
    for att in [(2, 0), (0, 4)]:
        assert hits[att][0] >= level_plane, hits
        assert hits[att][1] < level_sector, hits
