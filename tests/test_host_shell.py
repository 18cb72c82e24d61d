"""The C++ host mirror of the reference node classes (cones_perception_b200/host/nodes.hpp):
CPU tests of the stateful tracker, GPU tests of the full cloud_handlers."""
import ctypes as C
import os

import numpy as np
import pytest

from cones_perception_b200 import scans
from cones_perception_b200.build import HOST_LIB
from cones_perception_b200.params import PRESETS, GroundParams, to_c_detect
from oracle import oracle as O
from tests.util import TrackerReference

CAP = 256


@pytest.fixture(scope="module")
def host():
    lib = C.CDLL(HOST_LIB)
    lib.ch_last_error.restype = C.c_char_p
    lib.ch_tracker_create.restype = C.c_void_p
    lib.ch_tracker_create.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double]
    lib.ch_tracker_destroy.argtypes = [C.c_void_p]
    lib.ch_tracker_update.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32]
    lib.ch_detector_create.restype = C.c_void_p
    lib.ch_detector_create.argtypes = [C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.ch_detector_destroy.argtypes = [C.c_void_p]
    lib.ch_detector_handle.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ch_detector_set_color_inputs.argtypes = [C.c_void_p, C.c_int]
    lib.ch_detector_set_color_inputs.restype = None
    lib.ch_detector_load_color_model.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    lib.ch_detector_color_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ch_detector_color_probe.restype = None
    lib.ch_ground_create.restype = C.c_void_p
    lib.ch_ground_create.argtypes = [C.c_uint64, C.c_int]
    lib.ch_ground_destroy.argtypes = [C.c_void_p]
    lib.ch_ground_handle.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
    return lib


def tracker_update(lib, t, xy, forced=-1):
    xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
    out = np.zeros((4, CAP, 2), np.float32)
    counts = np.zeros(4, np.uint32)
    rc = lib.ch_tracker_update(t, xy.ctypes.data, len(xy), forced, out.ctypes.data, counts.ctypes.data, CAP)
    assert rc == 0
    return [out[k, :counts[k]].copy() for k in range(4)]


def as_arrays(clouds):
    return [np.array([(p[0], p[1]) for p in c], np.float32).reshape(-1, 2) for c in clouds]


@pytest.mark.parametrize("classify,buffer", [(False, False), (False, True), (True, True), (True, False)])
def test_tracker_matches_reference_semantics(host, classify, buffer):
    rng = np.random.default_rng(3)
    t = host.ch_tracker_create(int(classify), int(buffer), 0.5, 0.05)
    ref = TrackerReference(classify, buffer, 0.5, 0.05, forced_color=2)
    base = rng.uniform(1, 9, (12, 2)).astype(np.float32)
    for frame in range(8):
        # cones drift slowly, some appear / disappear, one frame is empty
        pts = base + rng.normal(0, 0.05 if frame % 3 else 0.4, base.shape).astype(np.float32)
        pts = pts[rng.random(len(pts)) > 0.2]
        if frame == 5:
            pts = pts[:0]
        got = tracker_update(host, t, pts, forced=2 if classify else -1)
        exp = as_arrays(ref.update([tuple(p) for p in pts]))
        for k in range(4):
            assert got[k].shape == exp[k].shape, (frame, k)
            assert np.array_equal(got[k].view(np.uint32), exp[k].view(np.uint32)), (frame, k)
        if frame == 0:
            assert sum(len(g) for g in got) == 0      # nothing is published on the first frame (Q8)
        if frame == 6 and not buffer and not classify:
            assert len(got[0]) == 0                   # previous frame detected nothing: gate stays shut
    host.ch_tracker_destroy(t)


@pytest.mark.gpu
@pytest.mark.parametrize("fused_ground,with_intensity", [(False, True), (True, True), (True, False)])
def test_cone_detector_cloud_handler_sequence(host, fused_ground, with_intensity):
    # a static scene seen 4 times with fresh sensor noise, so the temporal gate has matches:
    # cfg1 ("our" preset, level crop removes the ground) without, cfg2 with fused ground removal
    cfg = scans.config(2 if fused_ground else 1)
    frames = scans.generate(cfg, 4, base_seed=40)
    d = cfg.detect
    cd = to_c_detect(d)
    det = host.ch_detector_create(cfg.points_per_frame, 0, C.byref(cd), 0, 1, int(fused_ground))
    assert det, host.ch_last_error()
    ref = TrackerReference(False, True, d.cones_matching_dist_theshold, d.cone_position_extension_length)
    published = 0
    for f in frames:
        out = np.zeros((4, CAP, 2), np.float32)
        counts = np.zeros(4, np.uint32)
        step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
        rc = host.ch_detector_handle(det, f.ctypes.data, len(f), int(with_intensity), out.ctypes.data,
                                     counts.ctypes.data, CAP, C.byref(step), C.byref(nf), C.byref(nsec))
        assert rc == 0, host.ch_last_error()
        view = O.view_of_xyzi(f, with_intensity=True)
        if not with_intensity:
            view.off_intensity = 0                      # the faked field aliases x (src/cone_detection.cpp:142-151)
        cl, _, _ = O.detect(view, d, GroundParams() if fused_ground else None, O.CANONICAL)
        exp = as_arrays(ref.update([(c["x"], c["y"]) for c in cl]))
        for k in range(4):
            assert counts[k] == len(exp[k])
            assert np.array_equal(out[k, :counts[k]].view(np.uint32), exp[k].view(np.uint32))
        published += int(counts.sum())
        assert step.value == 32 and nf.value == (4 if with_intensity else 3)   # Q6: input fields, PCL data
        assert nsec.value == 123456789                                         # header copied verbatim
    assert published > 0
    host.ch_detector_destroy(det)


@pytest.mark.gpu
def test_cone_detector_colours_from_the_device_network(host):
    """classify_colors:=true with the classifier on the device (ConeDetector::load_color_model -> cp_cone_colors):
    the published colour clouds must equal the tracker driven by the CPU chain (reference box gather ->
    to_image -> numpy forward pass of dam_net -> 0.8 threshold) with the service's response semantics."""
    from cones_perception_b200 import tflite_model
    from oracle import dam_net_ref as D
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dam_net_model.npz")
    model = np.load(gold)["tflite"].tobytes()
    graph = tflite_model.load(model)
    cfg = scans.config(1)
    frames = scans.generate(cfg, 4, base_seed=40).copy()
    frames[..., 3] = np.clip(frames[..., 3] * 2.5, 0, 255)        # intensities in the range the network was trained on
    d = cfg.detect
    cd = to_c_detect(d)
    raw = {}

    def service(need):
        out = []
        for p in need:
            c = O.reconstruct_cone(raw["pts"], float(p[0]), float(p[1]), 0.228)
            if len(c) == 0:
                continue                                        # color_classifier_server.py:83-84
            img, fl = O.to_image(np.stack([c["x"], c["y"], c["z"], c["intensity"]], 1).astype(np.float32))
            if fl:
                return []                                       # to_image raises: the service call fails
            out.append(D.decide(D.forward(graph, img)[0]))
        return out

    det = host.ch_detector_create(cfg.points_per_frame, 0, C.byref(cd), 1, 1, 0)
    assert det, host.ch_last_error()
    buf = (C.c_uint8 * len(model)).from_buffer_copy(model)
    assert host.ch_detector_load_color_model(det, buf, len(model)) == 0, host.ch_last_error()
    ref = TrackerReference(True, True, d.cones_matching_dist_theshold, d.cone_position_extension_length,
                           color_fn=service)
    coloured = 0
    for f in frames:
        out = np.zeros((4, CAP, 2), np.float32)
        counts = np.zeros(4, np.uint32)
        step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
        rc = host.ch_detector_handle(det, f.ctypes.data, len(f), 1, out.ctypes.data, counts.ctypes.data, CAP,
                                     C.byref(step), C.byref(nf), C.byref(nsec))
        assert rc == 0, host.ch_last_error()
        raw["pts"] = O.from_msg(O.view_of_xyzi(f))
        cl, _, _ = O.detect(O.view_of_xyzi(f), d, None, O.CANONICAL)
        exp = as_arrays(ref.update([(c["x"], c["y"]) for c in cl]))
        for k in range(4):
            assert counts[k] == len(exp[k]), k
            assert np.array_equal(out[k, :counts[k]].view(np.uint32), exp[k].view(np.uint32))
        coloured += int(counts[1:].sum())
    assert coloured > 0
    host.ch_detector_destroy(det)


FNV0, FNVP, M64 = 1469598103934665603, 1099511628211, (1 << 64) - 1


def fnv1a(data: bytes, h: int = FNV0) -> int:
    for b in data:
        h = ((h ^ b) * FNVP) & M64
    return h


@pytest.mark.gpu
def test_cone_detector_colour_inputs_three_ways(host):
    """classify_colors:=true.  The colour-path inputs produced (0) by the reference's host loop, (1) by
    cp_cone_crops and (2) by cp_cone_images must drive the tracker identically; a deterministic stand-in
    for the classifier service (colour from a hash of its input, empty crops skipped) makes any differing
    crop or image change the published clouds."""
    cfg = scans.config(1)
    frames = scans.generate(cfg, 4, base_seed=40)
    frames[2] = frames[2].copy()
    d = cfg.detect
    cd = to_c_detect(d)
    raw = {}

    def crops_of(need):
        return [O.reconstruct_cone(raw["pts"], float(p[0]), float(p[1]), 0.228) for p in need]

    def colours_from_crops(need):
        out = []
        for c in crops_of(need):
            if len(c) == 0:
                continue
            h = fnv1a(np.stack([c["x"], c["y"], c["z"], c["intensity"]], 1).astype(np.float32).tobytes())
            raw["digest"] = fnv1a(h.to_bytes(8, "little"), raw["digest"])
            out.append(1 + h % 3)
        return out

    def colours_from_images(need):
        out = []
        for c in crops_of(need):
            img, fl = O.to_image(np.stack([c["x"], c["y"], c["z"], c["intensity"]], 1).astype(np.float32))
            if fl & O.CONE_EMPTY:
                continue
            h = fnv1a(img.tobytes())
            raw["digest"] = fnv1a(h.to_bytes(8, "little"), raw["digest"])
            out.append(1 + h % 3)
        return out

    results = []
    for mode in (0, 1, 2):
        det = host.ch_detector_create(cfg.points_per_frame, 0, C.byref(cd), 1, 1, 0)
        assert det, host.ch_last_error()
        host.ch_detector_set_color_inputs(det, mode)
        raw["digest"] = FNV0
        ref = TrackerReference(True, True, d.cones_matching_dist_theshold, d.cone_position_extension_length,
                               color_fn=colours_from_images if mode == 2 else colours_from_crops)
        seq = []
        for f in frames:
            out = np.zeros((4, CAP, 2), np.float32)
            counts = np.zeros(4, np.uint32)
            step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
            rc = host.ch_detector_handle(det, f.ctypes.data, len(f), 1, out.ctypes.data, counts.ctypes.data, CAP,
                                         C.byref(step), C.byref(nf), C.byref(nsec))
            assert rc == 0, host.ch_last_error()
            raw["pts"] = O.from_msg(O.view_of_xyzi(f))
            cl, _, _ = O.detect(O.view_of_xyzi(f), d, None, O.CANONICAL)
            exp = as_arrays(ref.update([(c["x"], c["y"]) for c in cl]))
            for k in range(4):
                assert counts[k] == len(exp[k]), (mode, k)
                assert np.array_equal(out[k, :counts[k]].view(np.uint32), exp[k].view(np.uint32))
            seq.append([out[k, :counts[k]].copy() for k in range(4)])
        n_in, n_pts, dig = C.c_uint64(), C.c_uint64(), C.c_uint64()
        host.ch_detector_color_probe(det, C.byref(n_in), C.byref(n_pts), C.byref(dig))
        assert dig.value == raw["digest"] and n_in.value > 5           # the service saw exactly these inputs
        results.append((seq, n_in.value, n_pts.value, dig.value))
        host.ch_detector_destroy(det)
    # host crops and GPU crops: identical service inputs, identical published clouds
    assert results[0][1:] == results[1][1:] and results[0][2] > 30
    for a, b in zip(results[0][0], results[1][0]):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert sum(len(c) for fr in results[2][0] for c in fr[1:]) > 0      # colours were assigned from images


@pytest.mark.gpu
def test_ground_remover_cloud_handler(host):
    cfg = scans.config(2)
    f = scans.generate(cfg, 1, base_seed=41)[0]
    gr = host.ch_ground_create(cfg.points_per_frame, 0)
    assert gr, host.ch_last_error()
    out = np.zeros((len(f), 8), np.float32)
    kept, step, nsec, nf = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
    rc = host.ch_ground_handle(gr, f.ctypes.data, len(f), 1, out.ctypes.data, C.byref(kept), C.byref(step),
                               C.byref(nsec), C.byref(nf))
    assert rc == 0, host.ch_last_error()
    exp, ekept, _, _ = O.ground_node(O.view_of_xyzi(f), GroundParams())
    e = np.stack([exp[n] for n in ("x", "y", "z", "pad", "intensity", "c1", "c2", "c3")], 1)
    assert kept.value == ekept and np.array_equal(out.view(np.uint32), e.view(np.uint32))
    assert step.value == 32 and nf.value == 4
    assert nsec.value == 123456000           # stamp survives the PCL round trip at microsecond resolution (Q5)
    host.ch_ground_destroy(gr)


@pytest.mark.gpu
@pytest.mark.parametrize("buffer", [True, False])
def test_cone_detector_matches_real_reference_node(host, buffer):
    """The C++ host mirror on the GPU library against the clouds the REAL cone_detection node published on the
    same 5-frame sequence (tests/golden/reference_nodes.npz, produced by the reference's own compiled source).
    Same cones frame by frame; centroids within north_star's 1e-5 m (PCL's voxel summation order is
    implementation-defined, the CUDA path uses the canonical one)."""
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_nodes.npz"))
    cfg = scans.config(1)
    cd = to_c_detect(cfg.detect)
    det = host.ch_detector_create(cfg.points_per_frame, 0, C.byref(cd), 0, int(buffer), 0)
    assert det, host.ch_last_error()
    for fi, f in enumerate(scans.generate(cfg, 5, base_seed=40)):
        out = np.zeros((4, CAP, 2), np.float32)
        counts = np.zeros(4, np.uint32)
        step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
        rc = host.ch_detector_handle(det, f.ctypes.data, len(f), 1, out.ctypes.data, counts.ctypes.data, CAP,
                                     C.byref(step), C.byref(nf), C.byref(nsec))
        assert rc == 0, host.ch_last_error()
        exp = z[f"detect_buffer{int(buffer)}_frame{fi}"]
        got = out[0, :counts[0]]
        assert got.shape == exp.shape and counts[1:].sum() == 0, fi
        if len(exp):
            assert np.allclose(got[np.lexsort(got.T)], exp[np.lexsort(exp.T)], rtol=0, atol=1e-5), fi
    host.ch_detector_destroy(det)


# ---- drop-in check at the message level: this repository's node shells behind the in-process ROS pump
# ---- (oracle/ref_shim) against what the reference's own nodes published for the same PointCloud2 messages

def _reference_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_nodes.npz"))


def _shell_lib():
    from cones_perception_b200.build import ROS_SHELL_LIB
    lib = C.CDLL(ROS_SHELL_LIB)
    vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int32
    lib.shell_last_error.restype = C.c_char_p
    lib.shell_ground_create.argtypes = [C.c_char_p]
    lib.shell_ground_create.restype = vp
    lib.shell_ground_destroy.argtypes = [vp]
    lib.shell_ground_handle.argtypes = [vp, vp, u32, u32, u32, u32, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.shell_ground_handle.restype = C.c_int64
    lib.shell_detect_create.argtypes = [C.c_char_p, C.c_int]
    lib.shell_detect_create.restype = vp
    lib.shell_detect_destroy.argtypes = [vp]
    lib.shell_detect_handle.argtypes = [vp, vp, u32, u32, u32, u32, i32, i32, i32, i32, vp, vp, u32, vp, vp]
    return lib


@pytest.mark.gpu
def test_ground_removal_node_shell_is_a_drop_in():
    """Same message into ros_shell/ground_removal_node.cpp on libconesgpu as into the reference's ground_removal
    node (its own source; what it published is stored in tests/golden/reference_nodes.npz): the published
    groundless_cloud must be identical — data bytes, point_step, field count, microsecond-truncated stamp."""
    import hashlib
    from tests.test_reference_pin import outside_sector_16
    z = _reference_golden()
    shell = _shell_lib()
    node = shell.shell_ground_create(b"")
    assert node, shell.shell_last_error()
    for seed in (0, 9):
        f = outside_sector_16(scans.generate(scans.config(2), 1, base_seed=seed)[0])
        assert hashlib.sha256(f.tobytes()).hexdigest() == str(z[f"ground_seed{seed}_input_sha256"])
        n = len(f)
        out = np.zeros((n, 8), np.float32)
        step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
        got = shell.shell_ground_handle(node, f.ctypes.data, n, 1, 16, 16 * n, 0, 4, 8, 12, out.ctypes.data,
                                        C.byref(step), C.byref(nf), C.byref(nsec))
        assert got == n
        assert np.array_equal(out[:256].view(np.uint32), z[f"ground_seed{seed}_head"].view(np.uint32))
        assert hashlib.sha256(out.tobytes()).hexdigest() == str(z[f"ground_seed{seed}_sha256"])
        assert (step.value, nf.value, nsec.value) == tuple(int(v) for v in z[f"ground_seed{seed}_meta"])
    shell.shell_ground_destroy(node)


@pytest.mark.gpu
@pytest.mark.parametrize("classify,buffer", [(False, True), (False, False), (True, True)])
def test_cone_detection_node_shell_is_a_drop_in(classify, buffer):
    """Same 5-message sequence into ros_shell/cone_detection_node.cpp as into the reference's cone_detection node:
    the same cones on the same four topics (centroids within north_star's 1e-5 m: PCL's voxel summation order is
    implementation-defined), same message layout.  With classify_colors the stand-in colour service hashes every
    crop it is sent, so the routing only matches if the crops do.  The reference's node runs live where its compiled
    library is present; without it, the cases without classify_colors use what the node published
    (tests/golden/reference_nodes.npz: the cones topic; nothing goes to the colour topics)."""
    from oracle import ref as R
    from tests.test_reference_pin import NO_NODES, node_params
    if classify and not R.available():
        pytest.skip(NO_NODES)
    cfg = scans.config(1)
    p = node_params(cfg.detect, classify_colors=classify, use_points_buffer=buffer)
    real = R.DetectNode(service=classify, **p) if R.available() else None
    z = _reference_golden()
    shell = _shell_lib()
    node = shell.shell_detect_create(R._params(p), 0 if classify else -1)
    assert node, shell.shell_last_error()
    total = 0
    for fi, f in enumerate(scans.generate(cfg, 5, base_seed=40)):
        exp = real.handle(f) if real else \
            [z[f"detect_buffer{int(buffer)}_frame{fi}"]] + [np.zeros((0, 2), np.float32)] * 3
        n = len(f)
        out = np.zeros((4, CAP, 2), np.float32)
        counts = np.zeros(4, np.uint32)
        step, nf = C.c_uint32(), C.c_uint32()
        rc = shell.shell_detect_handle(node, f.ctypes.data, n, 1, 16, 16 * n, 0, 4, 8, 12, out.ctypes.data,
                                       counts.ctypes.data, CAP, C.byref(step), C.byref(nf))
        assert rc == 0
        for k in range(4):
            got = out[k, :counts[k]]
            assert got.shape == exp[k].shape, (fi, k, counts.tolist(), [len(e) for e in exp])
            if len(got):
                assert np.allclose(got[np.lexsort(got.T)], exp[k][np.lexsort(exp[k].T)], rtol=0, atol=1e-5), (fi, k)
        total += int(counts.sum())
        if counts.sum():
            assert step.value == 32 and nf.value == 4
    assert total > 20
    if real:
        real.close()
    shell.shell_detect_destroy(node)
