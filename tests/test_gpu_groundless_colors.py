"""-m gpu: colour crops from the ground node's message after fused ground removal (cp_set_color_cloud GROUNDLESS).

In the reference's default launch the detection node crops colours from the ground node's groundless_cloud message:
the points the ground filter keeps, in input order, then N - G zero points.  Two references: the CPU chain
O.ground_node -> O.reconstruct_cone -> O.to_image -> dam_net_ref, and the two-handle device chain
(cp_batch_ground_remove to device memory, a second handle detecting on the 32-byte messages without ground removal,
then its colour call).  The fused run in GROUNDLESS mode must equal both, colours and probabilities bit for bit."""
import ctypes as C
import os

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200 import tflite_model as T
from cones_perception_b200.params import DetectParams, to_c_detect
from cones_perception_b200.pointcloud2 import PointCloud2, PointField
from oracle import dam_net_ref as D
from oracle import oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EXT = 0.05
UNSURE = api.CONE_AMBIGUOUS | api.CONE_LOW_CONFIDENCE
CFG2 = scans.config(2)
G = CFG2.ground


def _model() -> bytes:
    return np.load(os.path.join(GOLD, "dam_net_model.npz"))["tflite"].tobytes()


def _bright(frames):
    out = np.array(frames, np.float32, copy=True)
    out[..., 3] = np.clip(out[..., 3] * 2.5, 0, 255)
    return out


def _handle(max_points, max_frames, net=True, **kw):
    h = api.ConesGpu(max_points=max_points, max_frames=max_frames, **kw)
    if net:
        h.color_net_load_tflite(_model())
    return h


def _layout_msg(frame, step, offs):
    n = len(frame)
    raw = np.zeros((n, step), np.uint8)
    for k, o in enumerate(offs):
        raw[:, o:o + 4] = frame[:, k].copy().view(np.uint8).reshape(n, 4)
    names = ("x", "y", "z", "intensity")[:len(offs)]
    return PointCloud2(data=raw.reshape(-1), width=n, height=1, point_step=step,
                       fields=[PointField(nm, o) for nm, o in zip(names, offs)])


def _stage(h, frames, layout, keep):
    """Stage frames as the ground node reads them (no faked intensity)."""
    if layout == "device":
        import torch
        dev = torch.from_numpy(np.ascontiguousarray(np.concatenate(frames))).cuda()
        keep.append(dev)
        h.set_device_input(dev.data_ptr(), np.array([len(f) for f in frames], np.uint32), keep=dev)
    elif layout == "pcl32":
        h.set_host_input([_layout_msg(f, 32, (0, 4, 8, 16)) for f in frames], fake_missing_intensity=False)
    elif layout == "odd":
        h.set_host_input([_layout_msg(f, 22, (1, 5, 9, 14)) for f in frames], fake_missing_intensity=False)
    elif layout == "noint":
        h.set_host_input([_layout_msg(f, 12, (0, 4, 8)) for f in frames], fake_missing_intensity=False)
    else:
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames], fake_missing_intensity=False)


def _ground_msg(frame, with_intensity=True):
    return O.ground_node(O.view_of_xyzi(np.ascontiguousarray(frame, np.float32), with_intensity), G)[0]


def _cpu_chain(got, msg, clusters, net=True):
    """The service chain on the CPU, on the ground node's message of one frame."""
    g = T.load(_model())
    colors, probs, flags, counts = got
    for k, r in enumerate(clusters):
        cx, cy = O.extend(float(r["x"]), float(r["y"]), EXT)
        crop = O.reconstruct_cone(msg, cx, cy)
        assert int(counts[k]) == len(crop), k
        if len(crop) == 0:
            assert flags[k] & api.CONE_EMPTY and colors[k] == api.COLOR_NO_ANSWER, k
            continue
        img, fl = O.to_image(np.stack([crop["x"], crop["y"], crop["z"], crop["intensity"]], 1))
        if flags[k] & UNSURE:
            assert int(flags[k]) & ~UNSURE == fl, k
            continue
        assert int(flags[k]) == fl, k
        if fl:
            assert colors[k] == api.COLOR_NO_ANSWER, k
            continue
        if net:
            p, _ = D.forward(g, img)
            assert np.max(np.abs(p - probs[k])) <= 1e-6, k
            assert int(colors[k]) == D.decide(p), k


def _assert_same(got, ref):
    colors, probs, flags, counts = got
    assert np.array_equal(colors, ref[0])
    assert np.array_equal(probs.view(np.uint32), ref[1].view(np.uint32))
    assert np.array_equal(flags, ref[2])
    assert np.array_equal(counts, ref[3])


class Chain:
    """The reference's two-node launch on the device: handle a publishes the ground node's messages, handle b detects
    on them without ground removal and classifies from them."""

    def __init__(self, frames, layout="compact", detect=CFG2.detect):
        self.n = [len(f) for f in frames]
        total = max(sum(self.n), 1)
        self.keep = []
        self.a = api.ConesGpu(max_points=total, max_frames=len(frames), max_point_step=32)
        self.b = _handle(total, len(frames), max_point_step=32)
        self.detect = detect
        self.stage(frames, layout)

    def stage(self, frames, layout="compact"):
        self.n = [len(f) for f in frames]
        _stage(self.a, frames, layout, self.keep)
        self.a.batch_ground_remove(G, host=False)
        ptr, total = self.a.ground_device_output()
        assert total == sum(self.n)
        self.b.set_device_input(ptr, np.array(self.n, np.uint32), 32, (0, 4, 8, 16))
        self.b.run(self.detect, None)
        return self.b.results()

    def colors(self):
        return self.b.batch_cone_colors()

    def close(self):
        self.a.close()
        self.b.close()


def _fused(frames, layout="compact", detect=CFG2.detect, keep=None, **kw):
    h = _handle(max(sum(len(f) for f in frames), 1), len(frames), max_point_step=32, **kw)
    _stage(h, frames, layout, keep if keep is not None else [])
    h.run(detect, G)
    return h


def test_batch_colors_equal_the_cpu_chain():
    frames = _bright(scans.generate(CFG2, 16, base_seed=2040))
    with _fused(list(frames)) as h:
        _, off, cl = h.results()
        staged = h.batch_cone_colors()
        h.set_color_cloud(True)
        got = h.batch_cone_colors()
        assert len(cl) > 100
        for f in range(16):
            a, b = int(off[f]), int(off[f + 1])
            _cpu_chain(tuple(x[a:b] for x in got), _ground_msg(frames[f]), cl[a:b])
        # the ground returns around the cones are gone from the crops
        assert (got[3] != staged[3]).sum() > 0 and np.all(got[3] <= staged[3])
        answered = got[0][got[0] != api.COLOR_NO_ANSWER]
        assert len(set(answered.tolist())) >= 2


def _ragged():
    """config-1 frames: full, cut short, empty, no cluster (every point beyond the crop radius), full."""
    cfg = scans.config(1)
    src = _bright(scans.generate(cfg, 3, base_seed=2050))
    far = src[2].copy()
    far[:, :2] *= 100.0
    return cfg, [src[0], src[1][:17001], np.zeros((0, 4), np.float32), far, src[2]]


@pytest.mark.parametrize("layout", ["device", "compact", "pcl32", "odd"])
def test_batch_colors_equal_the_device_chain_every_layout(layout):
    cfg, frames = _ragged()
    chain = Chain(frames, layout, cfg.detect)
    keep = []
    try:
        _, coff, ccl = chain.b.results()
        exp = chain.colors()
        with _fused(frames, layout, cfg.detect, keep) as h:
            _, off, cl = h.results()
            assert np.array_equal(off, coff) and np.array_equal(cl.view(np.uint32), ccl.view(np.uint32))
            assert np.diff(off)[2] == 0 and np.diff(off)[3] == 0 and np.diff(off)[0] > 0
            h.set_color_cloud(True)
            _assert_same(h.batch_cone_colors(), exp)
    finally:
        chain.close()


@pytest.mark.parametrize("single", [True, False], ids=["single_launch", "single_off"])
def test_per_frame_calls_crop_the_ground_message(single):
    frame = _bright(scans.generate(CFG2, 1, base_seed=2060))[0]
    msg = _ground_msg(frame)
    kw = {} if single else {"env": {"CONESGPU_SINGLE": "0"}}
    with _handle(len(frame), 1, max_point_step=32, **kw) as h:
        h.set_color_cloud(True)
        cl, _ = h.detect(PointCloud2.from_xyzi(frame), CFG2.detect, G, fake_missing_intensity=False)
        if single:
            assert h.last_launch_count() == 1
        c = np.array([O.extend(float(r["x"]), float(r["y"]), EXT) for r in cl], np.float32)
        off, pts = h.cone_crops(c)
        for k, (cx, cy) in enumerate(c):
            exp = O.reconstruct_cone(msg, float(cx), float(cy))
            crop = pts[off[k]:off[k + 1]]
            assert len(crop) == len(exp), k
            e = np.stack([exp["x"], exp["y"], exp["z"], exp["intensity"]], 1)
            assert np.array_equal(crop.view(np.uint32), e.view(np.uint32)), k
        _, counts, flags = h.cone_images(c)
        colors, probs, flags2 = h.cone_colors(c)
        assert np.array_equal(counts, np.diff(off)) and np.array_equal(flags, flags2)
        _cpu_chain((colors, probs, flags2, counts), msg, cl)
        h.set_color_cloud(False)
        off_staged, _ = h.cone_crops(c)
        assert (np.diff(off_staged) > np.diff(off)).any()


def test_no_intensity_field():
    frames = list(_bright(scans.generate(CFG2, 4, base_seed=2070)))
    chain = Chain(frames, "noint")
    try:
        exp = chain.colors()
        with _fused(frames, "noint") as h:
            h.set_color_cloud(True)
            got = h.batch_cone_colors()
            _assert_same(got, exp)
            _, off, cl = h.results()
            for f in (0, 3):
                a, b = int(off[f]), int(off[f + 1])
                _cpu_chain(tuple(x[a:b] for x in got), _ground_msg(frames[f], with_intensity=False), cl[a:b])
            # per frame: every crop intensity is the ground node's 0
            h.detect(_layout_msg(frames[1], 12, (0, 4, 8)), CFG2.detect, G, fake_missing_intensity=False)
            _, off1, cl1 = h.results()
            c = np.array([O.extend(float(r["x"]), float(r["y"]), EXT) for r in cl1], np.float32)
            o, pts = h.cone_crops(c)
            assert o[-1] > 0 and not pts[:, 3].any()
            msg = _ground_msg(frames[1], with_intensity=False)
            e = np.concatenate([O.reconstruct_cone(msg, float(x), float(y)) for x, y in c])
            assert np.array_equal(pts.view(np.uint32), np.stack([e["x"], e["y"], e["z"], e["intensity"]], 1)
                                  .view(np.uint32))
    finally:
        chain.close()


def _near_sensor_frame(seed):
    """A config-2 frame plus a few points just ahead of the sensor, well above the ground: with no minimum distance
    and single-voxel clusters their cluster's extended box holds the origin, where the ground node pads."""
    f = _bright(scans.generate(CFG2, 1, base_seed=seed))[0]
    near = np.array([[0.06, 0.01, 0.3, 40.0], [0.061, 0.012, 0.31, 80.0], [0.07, -0.02, 0.35, 120.0]], np.float32)
    return np.concatenate([f[:5000], near, f[5000:]])


def test_padding_enters_a_crop_and_the_buffer_grows():
    d = DetectParams(**{**CFG2.detect.__dict__, "distance_treshold_min": 0.0, "min_cluster_size": 1})
    frames = [_near_sensor_frame(2080), _bright(scans.generate(CFG2, 1, base_seed=2081))[0]]
    msgs = [_ground_msg(f) for f in frames]
    chain = Chain(frames, detect=d)
    try:
        exp = chain.colors()
        with _fused(frames, detect=d) as h:        # a fresh handle: the crop buffer starts at 65 536 points
            ctr, off, cl = h.results()
            _, coff, ccl = chain.b.results()
            assert np.array_equal(off, coff) and np.array_equal(cl.view(np.uint32), ccl.view(np.uint32))
            h.set_color_cloud(True)
            got = h.batch_cone_colors()
            _assert_same(got, exp)
            pad = int(ctr["n_points"][0] - ctr["n_ground_kept"][0])
            assert pad > 65536
            at_origin = []
            for k in range(int(off[0]), int(off[1])):
                cx, cy = O.extend(float(cl[k]["x"]), float(cl[k]["y"]), EXT)
                crop = O.reconstruct_cone(msgs[0], cx, cy)
                assert got[3][k] == len(crop), k
                if abs(cx) <= 0.228 / 1.5 and abs(cy) <= 0.228 / 1.5:
                    at_origin.append((k, cx, cy, crop))
            assert at_origin
            _cpu_chain(tuple(x[int(off[0]):int(off[1])] for x in got), msgs[0], cl[int(off[0]):int(off[1])], net=False)
        with _handle(len(frames[0]), 1, max_point_step=32) as h:   # per-frame calls, fresh buffers
            h.set_color_cloud(True)
            cl0, ctr0 = h.detect(PointCloud2.from_xyzi(frames[0]), d, G, fake_missing_intensity=False)
            c = np.array([O.extend(float(r["x"]), float(r["y"]), EXT) for r in cl0], np.float32)
            _, counts, _ = h.cone_images(c)
            colors, _, flags = h.cone_colors(c)
            assert np.array_equal(counts, got[3][:len(c)]) and np.array_equal(colors, got[0][:len(c)])
            off1, pts = h.cone_crops(c, cap_points=int(counts.sum()))
            for k, _, _, crop in at_origin:
                seg = pts[off1[k]:off1[k + 1]]
                kept = len(crop) - pad
                assert kept > 0 and len(seg) == len(crop)
                assert not seg[kept:].any() and np.all(crop["x"][kept:] == 0)
                e = np.stack([crop["x"], crop["y"], crop["z"], crop["intensity"]], 1)
                assert np.array_equal(seg.view(np.uint32), e.view(np.uint32))
    finally:
        chain.close()


@pytest.mark.parametrize("buffer", [False, True])
def test_batch_track_equals_the_device_chain(buffer):
    frames = list(_bright(scans.generate(CFG2, 16, base_seed=2090)))
    seq = np.array([0, 3, 3, 8], np.uint32)
    p = api.track_params(True, buffer)
    chain = Chain(frames[:8])
    try:
        with _handle(8 * CFG2.points_per_frame, 8, max_point_step=32) as h:
            h.set_color_cloud(True)
            for half in (0, 1):                  # the second call continues the slots of the first
                part = frames[8 * half:8 * half + 8]
                if half:
                    chain.stage(part)
                _stage(h, part, "compact", [])
                h.run(CFG2.detect, G)
                ec, eo = chain.b.batch_track(p, seq)
                gc, go = h.batch_track(p, seq)
                assert np.array_equal(go, eo)
                assert gc.tobytes() == ec.tobytes() and len(gc) > 0
    finally:
        chain.close()


def test_run_without_ground_removal_is_unchanged():
    frames = list(_bright(scans.generate(CFG2, 4, base_seed=2100)))
    with _handle(4 * CFG2.points_per_frame, 4) as h:
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames])
        h.run(CFG2.detect, None)
        _, off, cl = h.results()
        staged = h.batch_cone_colors()
        c = np.array([O.extend(float(r["x"]), float(r["y"]), EXT) for r in cl[off[1]:off[2]]], np.float32)
        crops = h.cone_crops(c, frame=1)
        h.set_color_cloud(True)
        _assert_same(h.batch_cone_colors(), staged)
        g = h.cone_crops(c, frame=1)
        assert np.array_equal(g[0], crops[0]) and g[1].tobytes() == crops[1].tobytes()
        h.run(CFG2.detect, G)                                # a fused run in between
        h.batch_cone_colors()
        h.set_color_cloud(False)
        h.run(CFG2.detect, None)
        _assert_same(h.batch_cone_colors(), staged)


def _results_bytes(h):
    return b"".join(a.tobytes() for a in h.results())


@pytest.mark.parametrize("case", ["back_mode_3", "back_half_retry", "graph_replay", "no_rowskip"])
def test_robustness(case):
    if case == "back_half_retry":
        cfg = scans.config(4)
        frames = [_bright(scans.generate(cfg, 1, base_seed=0))[0]]   # dense: the shared-memory back half overflows
    else:
        cfg = CFG2
        frames = list(_bright(scans.generate(cfg, 4, base_seed=2110)))
    kw = {"back_mode": 3} if case == "back_mode_3" else {"env": {"CONESGPU_ROWSKIP": "0"}} if case == "no_rowskip" \
        else {}
    chain = Chain(frames, detect=cfg.detect)
    try:
        exp = chain.colors()
        with _handle(sum(len(f) for f in frames), len(frames), max_point_step=32, **kw) as h:
            h.set_color_cloud(True)
            _stage(h, frames, "compact", [])
            for _ in range(3 if case == "graph_replay" else 1):      # the third identical run replays a graph
                h.run(cfg.detect, G)
            st = h.lib.cp_batch_cone_colors(h._h, C.c_float(0.228), C.c_double(EXT), *[None] * 4, 0)
            assert st in (api.CP_OK, api.CP_E_CAPACITY)               # straight after the run: waits for it
            before = _results_bytes(h)
            got = h.batch_cone_colors()
            assert _results_bytes(h) == before
            _assert_same(got, exp)
            if case == "back_half_retry":
                e, _, _ = O.detect(O.view_of_xyzi(frames[0]), cfg.detect, G, O.CANONICAL)
                assert np.array_equal(h.results()[2].view(np.uint32), e.view(np.uint32))
    finally:
        chain.close()


def test_errors_and_launch_count():
    cfg = scans.config(3)
    frames = _bright(scans.generate(cfg, 64, base_seed=2120))
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    with _handle(64 * cfg.points_per_frame, 64) as h:
        for bad in (2, -1, 1 << 30):
            assert h.lib.cp_set_color_cloud(h._h, bad) == api.CP_E_PARAM
        h.set_color_cloud(True)
        h.set_host_input(msgs[:2])
        c = np.array([[5.0, 0.0]], np.float32)
        with pytest.raises(api.ConesGpuError) as e:               # staged, no run
            h.cone_crops(c)
        assert e.value.status == api.CP_E_STATE
        h.run(cfg.detect, G)
        h.cone_crops(c)
        h.set_host_input(msgs[2:4])                               # staged again since the run
        for call in (h.cone_crops, h.cone_images, h.cone_colors):
            with pytest.raises(api.ConesGpuError) as e:
                call(c)
            assert e.value.status == api.CP_E_STATE
        h.cone_crops(c, msg=msgs[0])                              # an explicit cloud is used as given
        launches = {}
        for n in (64, 8):
            h.set_host_input(msgs[:n])
            h.run(cfg.detect, G)
            h.batch_cone_colors()
            h.batch_cone_colors()
            launches[n] = h.last_launch_count()
        assert launches[8] == launches[64] > 0, launches
        h.set_color_cloud(False)
        h.batch_cone_colors()
        assert h.last_launch_count() == launches[8]


# ---- the C++ node layer --------------------------------------------------------------------------------------------
def _host_lib():
    from cones_perception_b200.build import HOST_LIB
    lib = C.CDLL(HOST_LIB)
    vp = C.c_void_p
    lib.ch_last_error.restype = C.c_char_p
    lib.ch_detector_create_replay.restype = vp
    lib.ch_detector_create_replay.argtypes = [C.c_uint64, C.c_uint32, C.c_int, vp, C.c_int, C.c_int, C.c_int]
    lib.ch_detector_destroy.argtypes = [vp]
    lib.ch_detector_publish.argtypes = [vp, vp, vp, C.c_uint32, C.c_int, C.c_int, vp, C.c_uint64,
                                        C.POINTER(C.c_uint64)]
    lib.ch_detector_set_color_inputs.argtypes = [vp, C.c_int]
    lib.ch_detector_set_color_inputs.restype = None
    lib.ch_detector_set_groundless_color_crops.argtypes = [vp, C.c_int]
    lib.ch_detector_set_groundless_color_crops.restype = None
    lib.ch_detector_load_color_model.argtypes = [vp, vp, C.c_uint64]
    lib.ch_detector_color_probe.argtypes = [vp, vp, vp, vp]
    lib.ch_detector_color_probe.restype = None
    lib.ch_ground_create.restype = vp
    lib.ch_ground_create.argtypes = [C.c_uint64, C.c_int]
    lib.ch_ground_destroy.argtypes = [vp]
    lib.ch_ground_handle.argtypes = [vp, vp, C.c_uint32, C.c_int, vp, vp, vp, vp, vp]
    return lib


def _cpp_publish(lib, det, frames, replay):
    xyzi = np.ascontiguousarray(np.concatenate(frames), np.float32)
    n = np.array([len(f) for f in frames], np.uint32)
    out = np.zeros(16 << 20, np.uint8)
    used = C.c_uint64()
    rc = lib.ch_detector_publish(det, xyzi.ctypes.data, n.ctypes.data, len(frames), 1, int(replay), out.ctypes.data,
                                 out.nbytes, C.byref(used))
    return rc, out[:used.value].tobytes()


def _cpp_ground(lib, frames):
    """GroundRemover::cloud_handler per message; the messages' x, y, z, intensity as compact clouds."""
    gr = lib.ch_ground_create(len(frames[0]), 0)
    out = []
    try:
        for f in frames:
            f = np.ascontiguousarray(f, np.float32)
            m = np.zeros((len(f), 8), np.float32)
            kept, step, stamp, nf = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
            assert lib.ch_ground_handle(gr, f.ctypes.data, len(f), 1, m.ctypes.data, C.byref(kept), C.byref(step),
                                        C.byref(stamp), C.byref(nf)) == 0, lib.ch_last_error()
            out.append(np.ascontiguousarray(m[:, [0, 1, 2, 4]]))
    finally:
        lib.ch_ground_destroy(gr)
    return out


@pytest.mark.parametrize("mode", ["gpu_crops", "gpu_colors", "replay", "host_crops"])
def test_cpp_detector_publishes_what_the_chained_nodes_publish(mode):
    lib = _host_lib()
    frames = list(_bright(scans.generate(CFG2, 4, base_seed=2130)))
    d = to_c_detect(CFG2.detect)
    n = CFG2.points_per_frame
    frames_per = 4 if mode == "replay" else 1
    fused = lib.ch_detector_create_replay(4 * n, frames_per, 0, C.byref(d), 1, 0, 1)
    plain = lib.ch_detector_create_replay(4 * n, frames_per, 0, C.byref(d), 1, 0, 0)
    try:
        assert fused and plain, lib.ch_last_error()
        lib.ch_detector_set_groundless_color_crops(fused, 1)
        for det in (fused, plain):
            if mode == "gpu_crops":
                lib.ch_detector_set_color_inputs(det, 1)          # hashing stand-in for the colour service
            elif mode == "host_crops":
                lib.ch_detector_set_color_inputs(det, 0)
            else:
                m = _model()
                assert lib.ch_detector_load_color_model(det, m, len(m)) == 0, lib.ch_last_error()
        if mode == "host_crops":
            rc, _ = _cpp_publish(lib, fused, frames, False)
            assert rc == 4 and b"kHostCrops" in lib.ch_last_error()
            return
        rc, got = _cpp_publish(lib, fused, frames, mode == "replay")
        assert rc == 0, lib.ch_last_error()
        rc, exp = _cpp_publish(lib, plain, _cpp_ground(lib, frames), mode == "replay")
        assert rc == 0, lib.ch_last_error()
        assert got == exp
        if mode == "gpu_crops":
            probes = []
            for det in (fused, plain):
                v = [C.c_uint64() for _ in range(3)]
                lib.ch_detector_color_probe(det, *[C.byref(x) for x in v])
                probes.append([x.value for x in v])
            assert probes[0] == probes[1] and probes[0][1] > 0
    finally:
        lib.ch_detector_destroy(fused)
        lib.ch_detector_destroy(plain)
