"""The plane ground model (cp_set_ground_plane) on the GPU, bit for bit against its CPU restatement
(oracle/plane_oracle.cpp; PARITY UNPINNED: the reference has no plane model).

A run with the plane model must equal the two-node chain of the oracle: the plane ground node's message, then the
detector without ground removal on it.  Every case compares the hypothesis and count taps, the chosen planes, their
inliers and indices, the counters, the cluster offsets and the records; the ground calls compare the messages byte for
byte."""
import ctypes as C

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200.params import GroundParams, to_c_ground
from cones_perception_b200.pointcloud2 import PointCloud2
from oracle import oracle as O
from oracle import plane_oracle as PO
from tests.test_gpu_parity import _msg_with_layout

P = PO.PlaneParams(seed=1, n_hypotheses=64, inlier_distance=0.1, ground_height=0.1, max_tilt_deg=15.0)
G = GroundParams()
CFG3 = scans.config(3)
FIELDS = ("x", "y", "z", "pad", "intensity", "c1", "c2", "c3")
CTR = ("n_points", "n_ground_kept", "n_cropped", "n_voxels", "n_components", "n_clusters")


def _rotate(p, pitch_deg, roll_deg):
    a, b = np.radians(pitch_deg), np.radians(roll_deg)
    Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    Rx = np.array([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]])
    q = p.astype(np.float64)
    q[:, :3] = q[:, :3] @ (Rx @ Ry).T
    return np.ascontiguousarray(q.astype(np.float32))


def _pitched(n, seed=0, cfg=CFG3):
    rng = np.random.default_rng(seed)
    return [_rotate(f, *rng.uniform(-3, 3, 2)) for f in scans.generate(cfg, n, base_seed=seed)]


def _expect(records, p=P, d=CFG3.detect):
    """Per frame from the oracle: hypotheses, counts, (plane, inliers, hypothesis), message bytes, kept, clusters,
    counters."""
    out = []
    for r in records:
        hyp = PO.hypotheses(r, p)
        cnt = PO.counts(r, hyp, p.inlier_distance)
        msg, kept, plane, inl, h, _ = PO.ground_node(r, p)
        cl, ctr, _ = O.detect(PO.view_of_records(msg), d, None, O.CANONICAL)
        mb = np.stack([msg[n] for n in FIELDS], 1).astype(np.float32).tobytes() if len(msg) else b""
        out.append(dict(hyp=hyp, cnt=cnt, plane=plane, inl=inl, h=h, msg=mb, kept=kept, cl=cl,
                        ctr={k: getattr(ctr, k) for k in CTR} | {"n_ground_kept": kept}))
    return out


def _records(msgs, fake_missing_intensity):
    return [O.from_msg(O.view_of_msg(m, fake_missing_intensity)) for m in msgs]


def _check_planes(h, exp, p=P):
    F, H = len(exp), p.n_hypotheses
    hyp = h.tap(api.TAP_PLANE_HYPOTHESES).reshape(F, H, 4)
    cnt = h.tap(api.TAP_PLANE_COUNTS).reshape(F, H)
    planes, inl, hi = h.ground_planes()
    for f, e in enumerate(exp):
        assert np.array_equal(hyp[f].view(np.uint32), e["hyp"].view(np.uint32)), f"frame {f}: hypotheses"
        assert np.array_equal(cnt[f], e["cnt"]), f"frame {f}: counts"
        assert np.array_equal(planes[f].view(np.uint32), e["plane"].view(np.uint32)), f"frame {f}: plane"
        assert (int(inl[f]), int(hi[f])) == (e["inl"], e["h"]), f"frame {f}"


def _check_run(h, exp, p=P):
    ctr, off, cl = h.results()
    _check_planes(h, exp, p)
    for f, e in enumerate(exp):
        got = cl[off[f]:off[f + 1]]
        assert np.array_equal(got.view(np.uint32), e["cl"].view(np.uint32)), f"frame {f}: clusters"
        for k, v in e["ctr"].items():
            assert int(ctr[k][f]) == v, (f, k, int(ctr[k][f]), v)
    return ctr, off, cl


def _check_ground(h, exp):
    out, kept, low = h.batch_ground_remove(G)
    assert low is None
    raw = out.tobytes()
    at = 0
    for f, e in enumerate(exp):
        assert raw[at:at + len(e["msg"])] == e["msg"], f"frame {f}: message"
        assert int(kept[f]) == e["kept"]
        at += len(e["msg"])
    _check_planes(h, exp)
    return out


@pytest.mark.gpu
def test_pitched_batch_graph_replay_and_model_switch():
    frames = _pitched(64, seed=3)
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    exp = _expect(_records(msgs, True))
    total = sum(len(f) for f in frames)
    with api.ConesGpu(max_points=total, max_frames=len(frames)) as h:
        h.set_host_input(msgs)
        h.set_ground_plane(P)
        for _ in range(3):   # the second identical run is captured, the third replays the graph
            h.run(CFG3.detect, G)
            _check_run(h, exp)
        # sector -> plane -> sector on one staged input
        h.set_ground_plane(None)
        h.run(CFG3.detect, G)
        ctr, off, cl = h.results()
        for f in (0, 31, 63):
            e, octr, _ = O.detect(O.view_of_msg(msgs[f], True), CFG3.detect, G, O.CANONICAL)
            assert np.array_equal(cl[off[f]:off[f + 1]].view(np.uint32), e.view(np.uint32))
            assert int(ctr["n_ground_kept"][f]) == octr.n_ground_kept
        with pytest.raises(api.ConesGpuError) as ei:
            h.ground_planes()
        assert ei.value.status == api.CP_E_STATE
        h.set_ground_plane(P)
        h.run(CFG3.detect, G)
        _check_run(h, exp)
        assert h.last_rows_loaded() == sum((len(f) + 31) // 32 for f in frames)   # no row is skipped


def _ragged_frames():
    cfg = scans.config(2)
    src = scans.generate(cfg, 2, base_seed=40)
    nan = src[0][:700].copy()
    nan[:, 2] = np.nan
    line = np.zeros((900, 4), np.float32)                      # collinear: every hypothesis degenerate
    line[:, 0] = np.linspace(1, 9, 900, dtype=np.float32)
    line[:, 2] = -0.6
    frames = [src[0], np.zeros((0, 4), np.float32), src[1][:1], src[1][:2], src[1][:3], src[1][5000:5000 + 2049],
              nan, line, _rotate(src[1], 0, 0)]
    return [np.ascontiguousarray(f, np.float32) for f in frames]


@pytest.mark.gpu
@pytest.mark.parametrize("level", [True, False])
def test_level_and_ragged_frames(level):
    frames = _ragged_frames() if not level else [np.ascontiguousarray(f) for f in scans.generate(CFG3, 6, 8)]
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    exp = _expect(_records(msgs, True))
    gexp = _expect(_records(msgs, False))
    total = sum(len(f) for f in frames)
    with api.ConesGpu(max_points=total, max_frames=len(frames)) as h:
        h.set_ground_plane(P)
        h.set_host_input(msgs)
        h.run(CFG3.detect, G)
        _check_run(h, exp)
        h.set_host_input(msgs, fake_missing_intensity=False)
        _check_ground(h, gexp)
    if not level:
        assert exp[1]["h"] == exp[2]["h"] == exp[3]["h"] == -1 and exp[4]["kept"] <= 3
        assert exp[6]["kept"] == 0 and exp[7]["h"] == -1 and exp[7]["kept"] == 900


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["compact", "pcl32", "unaligned22", "no_intensity", "device"])
def test_layouts(layout):
    frames = _pitched(4, seed=11)
    fx = [f[:120_000] for f in frames]
    if layout == "compact":
        msgs = [PointCloud2.from_xyzi(f) for f in fx]
    elif layout == "pcl32":
        msgs = [_msg_with_layout(f, 32, (0, 4, 8, 16)) for f in fx]
    elif layout == "unaligned22":
        msgs = [_msg_with_layout(f, 22, (0, 4, 8, 12)) for f in fx]
    else:
        msgs = [_msg_with_layout(f, 16, (0, 4, 8, 12), intensity=False) for f in fx]
    total = sum(len(f) for f in fx)
    with api.ConesGpu(max_points=total, max_frames=4, max_point_step=32) as h:
        h.set_ground_plane(P)
        if layout == "device":
            import torch
            dev = torch.from_numpy(np.ascontiguousarray(np.concatenate(fx))).cuda()
            h.set_device_input(dev.data_ptr(), [len(f) for f in fx], 16, (0, 4, 8, 12), keep=dev)
            exp = _expect(fx)
        else:
            h.set_host_input(msgs)
            exp = _expect(_records(msgs, True))
        h.run(CFG3.detect, G)
        _check_run(h, exp)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["cfg4_retry", "cfg5", "back_mode3", "single0"])
def test_back_half_paths(case):
    env = {}
    p = P
    if case == "cfg4_retry":
        # a plane that keeps every point: the config-4 frame's survivors overflow the per-frame back half
        cfg = scans.config(4)
        frames = [scans.generate(cfg, 1, base_seed=2)[0]]
        p = PO.PlaneParams(**{**P.__dict__, "ground_height": -1000.0})
    elif case == "cfg5":
        cfg = scans.config(5)
        frames = _pitched(3, seed=5, cfg=cfg)
    else:
        cfg = CFG3
        frames = _pitched(3, seed=6)
        env = {"CONESGPU_BACK_MODE": "3"} if case == "back_mode3" else {"CONESGPU_SINGLE": "0"}
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    exp = _expect(_records(msgs, True), p=p, d=cfg.detect)
    total = sum(len(f) for f in frames)
    with api.ConesGpu(max_points=total, max_frames=len(frames), env=env) as h:
        h.set_ground_plane(p)
        h.set_host_input(msgs)
        h.run(cfg.detect, G)
        before = h.last_launch_count()
        h.sync()
        if case == "cfg4_retry":
            assert h.last_launch_count() > before, "cp_sync did not re-run the back half"
        _check_run(h, exp, p)
        # the single-frame call on each frame equals the batch frame
        for f, m in enumerate(msgs):
            got, ctr = h.detect(m, cfg.detect, G)
            assert np.array_equal(np.asarray(got).view(np.uint32), exp[f]["cl"].view(np.uint32))
            assert int(ctr["n_ground_kept"]) == exp[f]["kept"]


@pytest.mark.gpu
def test_position_batch_size_and_seed():
    frames = _pitched(8, seed=21)
    with api.ConesGpu(max_points=sum(len(f) for f in frames), max_frames=8) as h:
        h.set_ground_plane(P)
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames])
        h.run(CFG3.detect, G)
        ctr8, off8, cl8 = h.results()
        hyp8 = h.tap(api.TAP_PLANE_HYPOTHESES).reshape(8, -1, 4)
        planes8 = h.ground_planes()
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames[5:6]])
        h.run(CFG3.detect, G)
        ctr1, off1, cl1 = h.results()
        assert np.array_equal(h.tap(api.TAP_PLANE_HYPOTHESES).reshape(-1, 4).view(np.uint32), hyp8[5].view(np.uint32))
        assert np.array_equal(cl1.view(np.uint32), cl8[off8[5]:off8[6]].view(np.uint32))
        assert np.array_equal(h.ground_planes()[0].view(np.uint32), planes8[0][5:6].view(np.uint32))
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames[::-1]])   # frame 5 now sits at position 2
        h.run(CFG3.detect, G)
        ctr, off, cl = h.results()
        assert np.array_equal(cl[off[2]:off[3]].view(np.uint32), cl8[off8[5]:off8[6]].view(np.uint32))
        q = PO.PlaneParams(**{**P.__dict__, "seed": 2})
        h.set_ground_plane(q)
        h.run(CFG3.detect, G)
        other = h.tap(api.TAP_PLANE_HYPOTHESES).reshape(8, -1, 4)
        assert not np.array_equal(other[2].view(np.uint32), hyp8[5].view(np.uint32))
        assert np.array_equal(other[2].view(np.uint32), PO.hypotheses(frames[5], q).view(np.uint32))


@pytest.mark.gpu
def test_device_two_node_chain_equals_fused_run():
    frames = _pitched(5, seed=31)
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    n = [len(f) for f in frames]
    with api.ConesGpu(max_points=sum(n), max_frames=5, max_point_step=32) as a, \
            api.ConesGpu(max_points=sum(n), max_frames=5, max_point_step=32) as b:
        a.set_ground_plane(P)
        a.set_host_input(msgs, fake_missing_intensity=False)
        _, kept, _ = a.batch_ground_remove(G, host=False)
        ptr, total = a.ground_device_output()
        b.set_device_input(ptr, n, 32, (0, 4, 8, 16))
        b.run(CFG3.detect)
        ctr_b, off_b, cl_b = b.results()
        a.run(CFG3.detect, G)
        ctr_a, off_a, cl_a = a.results()
    assert np.array_equal(off_a, off_b) and np.array_equal(cl_a.view(np.uint32), cl_b.view(np.uint32))
    assert np.array_equal(ctr_a["n_ground_kept"], kept)
    for k in CTR:
        if k != "n_ground_kept":
            assert np.array_equal(ctr_a[k], ctr_b[k]), k


@pytest.mark.gpu
def test_errors_and_launch_counts():
    frames = _pitched(2, seed=41)
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    with api.ConesGpu(max_points=sum(len(f) for f in frames), max_frames=2) as h:
        lib = h.lib
        for bad in (dict(n_hypotheses=0), dict(n_hypotheses=257), dict(inlier_distance=0.0),
                    dict(inlier_distance=float("nan")), dict(ground_height=float("inf")), dict(max_tilt_deg=0.0),
                    dict(max_tilt_deg=90.5)):
            c = api.plane_params(**bad)
            assert lib.cp_set_ground_plane(h._h, C.byref(c)) == api.CP_E_PARAM, bad
        assert lib.cp_set_ground_plane(h._h, C.byref(api.plane_params(max_tilt_deg=90.0))) == api.CP_OK
        h.set_host_input(msgs)
        h.run(CFG3.detect, G)
        with pytest.raises(api.ConesGpuError) as ei:
            h.tap(api.TAP_SECTOR_LOW)
        assert ei.value.status == api.CP_E_STATE
        assert lib.cp_ground_planes(h._h, None, None, None, 1) == api.CP_E_CAPACITY
        assert lib.cp_ground_planes(h._h, None, None, None, 2) == api.CP_OK
        # colour crops from the groundless cloud re-derive the sector verdict: refused after a plane run
        h.set_color_cloud(True)
        centers = np.full(2, 1000.0, np.float32)   # a box far from every point
        offs = np.zeros(2, np.uint32)
        assert lib.cp_cone_crops(h._h, None, 0, centers.ctypes.data, 1, 0.228, offs.ctypes.data, None, 0) == \
            api.CP_E_STATE
        h.set_color_cloud(False)
        assert lib.cp_cone_crops(h._h, None, 0, centers.ctypes.data, 1, 0.228, offs.ctypes.data, None, 0) == api.CP_OK
        # low17 under the plane model
        g = to_c_ground(G)
        low = np.zeros(34, np.float32)
        kept = np.zeros(2, np.uint32)
        assert lib.cp_batch_ground_remove(h._h, C.byref(g), None, 0, kept.ctypes.data, low.ctypes.data) == \
            api.CP_E_PARAM
        h.set_ground_plane(None)
        h.run(CFG3.detect, G)
        assert lib.cp_ground_planes(h._h, None, None, None, 2) == api.CP_E_STATE
    counts = []
    small = [f[:4000] for f in _pitched(8, seed=51)]
    for F in (8, 512):
        fr = [small[i % 8] for i in range(F)]
        with api.ConesGpu(max_points=sum(len(f) for f in fr), max_frames=F) as h:
            h.set_ground_plane(P)
            h.set_host_input([PointCloud2.from_xyzi(f) for f in fr])
            h.run(CFG3.detect, G)
            h.sync()
            counts.append(h.last_launch_count())
            h.batch_ground_remove(G)
            counts.append(h.last_launch_count())
    assert counts[0] == counts[2] and counts[1] == counts[3], counts


@pytest.mark.gpu
def test_graph_replay_around_a_ground_call():
    """plane run x 2 (the second is captured), a ground call, then runs again: each run's results, the taps and the
    refusal of groundless colour crops must describe the plane chain, whether the run was enqueued or replayed."""
    frames = _pitched(4, seed=61)
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    gexp = _expect(_records(msgs, False))
    centers = np.full(2, 1000.0, np.float32)
    offs = np.zeros(2, np.uint32)
    with api.ConesGpu(max_points=sum(len(f) for f in frames), max_frames=4) as h:
        h.set_ground_plane(P)
        h.set_color_cloud(True)
        h.set_host_input(msgs, fake_missing_intensity=False)
        for step in range(5):
            if step == 2:
                _check_ground(h, gexp)
            h.run(CFG3.detect, G)
            _check_run(h, gexp)
            assert h.lib.cp_cone_crops(h._h, None, 0, centers.ctypes.data, 1, 0.228, offs.ctypes.data, None, 0) == \
                api.CP_E_STATE, step


def _host_lib():
    from cones_perception_b200.build import HOST_LIB
    lib = C.CDLL(HOST_LIB)
    vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int
    lib.ch_last_error.restype = C.c_char_p
    lib.ch_ground_create.restype = vp
    lib.ch_ground_create.argtypes = [C.c_uint64, i32]
    lib.ch_ground_create_replay.restype = vp
    lib.ch_ground_create_replay.argtypes = [C.c_uint64, u32, i32]
    lib.ch_ground_destroy.argtypes = [vp]
    lib.ch_ground_handle.argtypes = [vp, vp, u32, i32, vp, vp, vp, vp, vp]
    lib.ch_ground_publish.argtypes = [vp, vp, vp, u32, i32, i32, vp, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.ch_detector_create.restype = vp
    lib.ch_detector_create.argtypes = [C.c_uint64, i32, vp, i32, i32, i32]
    lib.ch_detector_create_replay.restype = vp
    lib.ch_detector_create_replay.argtypes = [C.c_uint64, u32, i32, vp, i32, i32, i32]
    lib.ch_detector_destroy.argtypes = [vp]
    lib.ch_detector_publish.argtypes = [vp, vp, vp, u32, i32, i32, vp, C.c_uint64, C.POINTER(C.c_uint64)]
    for f in (lib.ch_ground_set_ground_model, lib.ch_detector_set_ground_model):
        f.argtypes = [vp, i32, i32, i32, C.c_double, C.c_double, C.c_double]
        f.restype = None
    return lib


def _set_plane(fn, obj, p=P):
    fn(obj, 1, p.seed, p.n_hypotheses, p.inlier_distance, p.ground_height, p.max_tilt_deg)


def _publish(fn, obj, frames, replay):
    xyzi = np.ascontiguousarray(np.concatenate(frames), np.float32)
    n = np.array([len(f) for f in frames], np.uint32)
    out = np.zeros(64 << 20, np.uint8)
    used = C.c_uint64()
    assert fn(obj, xyzi.ctypes.data, n.ctypes.data, len(frames), 1, int(replay), out.ctypes.data, out.nbytes,
              C.byref(used)) == 0
    return out[:used.value].tobytes()


@pytest.mark.gpu
def test_cpp_nodes_against_the_oracle():
    """The C++ GroundRemover with ground_model = "plane" publishes the oracle's messages (cloud_handler and replay);
    the ConeDetector fusing the plane ground removal publishes what a detector without ground removal publishes on
    the oracle's messages (cloud_handler and replay)."""
    from cones_perception_b200.params import to_c_detect
    lib = _host_lib()
    frames = _pitched(5, seed=71)
    n = CFG3.points_per_frame
    gr = lib.ch_ground_create(n, 0)
    grr = lib.ch_ground_create_replay(2 * n, 2, 0)
    cd = to_c_detect(CFG3.detect)
    fused = lib.ch_detector_create(n, 0, C.byref(cd), 0, 0, 1)
    fused_replay = lib.ch_detector_create_replay(2 * n, 2, 0, C.byref(cd), 0, 0, 1)
    plain = lib.ch_detector_create(n, 0, C.byref(cd), 0, 0, 0)
    try:
        assert gr and grr and fused and fused_replay and plain, lib.ch_last_error()
        for obj in (gr, grr):
            _set_plane(lib.ch_ground_set_ground_model, obj)
        for obj in (fused, fused_replay):
            _set_plane(lib.ch_detector_set_ground_model, obj)
        msgs_xyzi = []
        for f in frames:
            msg, kept, _, _, _, _ = PO.ground_node(f, P)
            out = np.zeros((len(f), 8), np.float32)
            k, step, nsec, nf = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
            assert lib.ch_ground_handle(gr, f.ctypes.data, len(f), 1, out.ctypes.data, C.byref(k), C.byref(step),
                                        C.byref(nsec), C.byref(nf)) == 0, lib.ch_last_error()
            exp = np.stack([msg[c] for c in FIELDS], 1).astype(np.float32)
            assert out.tobytes() == exp.tobytes() and k.value == kept
            msgs_xyzi.append(np.ascontiguousarray(np.stack([msg["x"], msg["y"], msg["z"], msg["intensity"]], 1)))
        assert _publish(lib.ch_ground_publish, grr, frames, True) == _publish(lib.ch_ground_publish, gr, frames, False)
        exp = _publish(lib.ch_detector_publish, plain, msgs_xyzi, False)
        assert _publish(lib.ch_detector_publish, fused, frames, False) == exp
        assert _publish(lib.ch_detector_publish, fused_replay, frames, True) == exp
    finally:
        for obj in (gr, grr):
            lib.ch_ground_destroy(obj)
        for obj in (fused, fused_replay, plain):
            lib.ch_detector_destroy(obj)


@pytest.mark.gpu
def test_ros_ground_shell_reads_the_plane_parameters():
    from tests.test_host_shell import _shell_lib
    shell = _shell_lib()
    params = (f"~ground_model=plane;~plane_seed={P.seed};~plane_hypotheses={P.n_hypotheses};"
              f"~plane_inlier_distance={P.inlier_distance!r};~plane_ground_height={P.ground_height!r};"
              f"~plane_max_tilt_deg={P.max_tilt_deg!r}").encode()
    node = shell.shell_ground_create(params)
    assert node, shell.shell_last_error()
    try:
        for f in _pitched(2, seed=81):
            n = len(f)
            out = np.zeros((n, 8), np.float32)
            step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
            got = shell.shell_ground_handle(node, f.ctypes.data, n, 1, 16, 16 * n, 0, 4, 8, 12, out.ctypes.data,
                                            C.byref(step), C.byref(nf), C.byref(nsec))
            msg, kept, _, _, _, _ = PO.ground_node(f, P)
            assert got == n
            assert out.tobytes() == np.stack([msg[c] for c in FIELDS], 1).astype(np.float32).tobytes()
            assert kept < n
    finally:
        shell.shell_ground_destroy(node)
