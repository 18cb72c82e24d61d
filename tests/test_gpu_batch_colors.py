"""-m gpu: colours for every cluster of a batch run (cp_batch_cone_colors), bit for bit.

Two references: cp_cone_colors on the same handle, one frame at a time, at the centres the node would pass
(O.extend of each record); and the CPU chain O.reconstruct_cone -> O.to_image -> dam_net_ref.forward / decide.
Colours, flags and counts must be equal; probabilities equal as uint32 against the per-frame call (the same device
arithmetic) and within 1e-6 against the numpy network.  Intensities are scaled into the range the network was
trained on so that several colours occur."""
import ctypes as C
import os

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200 import tflite_model as T
from cones_perception_b200.pointcloud2 import PointCloud2, PointField
from oracle import dam_net_ref as D
from oracle import oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EXT = 0.05
UNSURE = api.CONE_AMBIGUOUS | api.CONE_LOW_CONFIDENCE


def _model() -> bytes:
    return np.load(os.path.join(GOLD, "dam_net_model.npz"))["tflite"].tobytes()


def _bright(frames):
    out = np.array(frames, np.float32, copy=True)
    out[..., 3] = np.clip(out[..., 3] * 2.5, 0, 255)
    return out


def _handle(max_points, max_frames, **kw):
    h = api.ConesGpu(max_points=max_points, max_frames=max_frames, **kw)
    h.color_net_load_tflite(_model())
    return h


def _per_frame(h, clusters, off, ext=EXT):
    """cp_cone_colors frame by frame on the handle's staged input, centres extended as the node does."""
    K = len(clusters)
    colors, flags, counts = np.zeros(K, np.uint8), np.zeros(K, np.uint32), np.zeros(K, np.uint32)
    probs = np.zeros((K, 3), np.float32)
    for f in range(len(off) - 1):
        a, b = int(off[f]), int(off[f + 1])
        if a == b:
            continue
        c = np.array([O.extend(float(r["x"]), float(r["y"]), ext) for r in clusters[a:b]], np.float32)
        colors[a:b], probs[a:b], flags[a:b] = h.cone_colors(c, frame=f)
        _, counts[a:b], _ = h.cone_images(c, frame=f)
    return colors, probs, flags, counts


def _assert_same(got, ref):
    colors, probs, flags, counts = got
    assert np.array_equal(colors, ref[0])
    assert np.array_equal(probs.view(np.uint32), ref[1].view(np.uint32))
    assert np.array_equal(flags, ref[2])
    assert np.array_equal(counts, ref[3])


def _assert_cpu_chain(got, frame, clusters, ext=EXT):
    """The service chain on the CPU for one frame's clusters."""
    g = T.load(_model())
    pts = O.points32(frame)
    colors, probs, flags, counts = got
    for k, r in enumerate(clusters):
        cx, cy = O.extend(float(r["x"]), float(r["y"]), ext)
        crop = O.reconstruct_cone(pts, cx, cy)
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
        p, _ = D.forward(g, img)
        assert np.max(np.abs(p - probs[k])) <= 1e-6, k
        assert int(colors[k]) == D.decide(p), k


def _oracle_counts(frame, clusters, ext=EXT):
    pts = O.points32(frame)
    return np.array([len(O.reconstruct_cone(pts, *O.extend(float(r["x"]), float(r["y"]), ext)))
                     for r in clusters], np.uint32)


def test_batch_colors_match_per_frame_and_cpu_chain():
    cfg = scans.config(2)
    frames = _bright(scans.generate(cfg, 16, base_seed=40))
    with _handle(16 * cfg.points_per_frame, 16) as h:
        _, off, cl = h.detect_batch([PointCloud2.from_xyzi(f) for f in frames], cfg.detect, cfg.ground)
        got = h.batch_cone_colors()
        assert len(got[0]) == len(cl) > 100
        _assert_same(got, _per_frame(h, cl, off))
        for f in range(16):
            a, b = int(off[f]), int(off[f + 1])
            assert np.array_equal(got[3][a:b], _oracle_counts(frames[f], cl[a:b])), f
        for f in (0, 15):
            a, b = int(off[f]), int(off[f + 1])
            _assert_cpu_chain(tuple(x[a:b] for x in got), frames[f], cl[a:b])
        answered = got[0][got[0] != api.COLOR_NO_ANSWER]
        assert len(set(answered.tolist())) >= 2


def _ragged_frames():
    """Five config-1 frames: full, cut short, empty, no cluster (every point beyond the crop radius), full."""
    cfg = scans.config(1)
    src = _bright(scans.generate(cfg, 3, base_seed=50))
    far = src[2].copy()
    far[:, :2] *= 100.0
    return cfg, [src[0], src[1][:17001], np.zeros((0, 4), np.float32), far, src[2]]


def _layout_msg(frame, step, offs):
    n = len(frame)
    raw = np.zeros((n, step), np.uint8)
    for k, o in enumerate(offs):
        raw[:, o:o + 4] = frame[:, k].copy().view(np.uint8).reshape(n, 4)
    return PointCloud2(data=raw.reshape(-1), width=n, height=1, point_step=step,
                       fields=[PointField(nm, o) for nm, o in zip(("x", "y", "z", "intensity"), offs)])


@pytest.mark.parametrize("layout", ["device", "pcl32", "odd"])
def test_batch_colors_every_input_layout(layout):
    cfg, frames = _ragged_frames()
    total = sum(len(f) for f in frames)
    with _handle(total, len(frames), max_point_step=32) as h:
        if layout == "device":          # layout mode 0: compact float4, caller's device memory
            import torch
            dev = torch.from_numpy(np.ascontiguousarray(np.concatenate(frames))).cuda()
            h.set_device_input(dev.data_ptr(), np.array([len(f) for f in frames], np.uint32), keep=dev)
        elif layout == "pcl32":         # mode 1: x@0 y@4 z@8 intensity@16, step 32
            h.set_host_input([_layout_msg(f, 32, (0, 4, 8, 16)) for f in frames])
        else:                           # mode 2: unaligned fields, byte-wise loads
            h.set_host_input([_layout_msg(f, 23, (1, 5, 9, 14)) for f in frames])
        h.run(cfg.detect, cfg.ground)
        _, off, cl = h.results()
        counts_per_frame = np.diff(off)
        assert counts_per_frame[2] == 0 and counts_per_frame[3] == 0
        assert counts_per_frame[0] > 0 and counts_per_frame[1] > 0 and counts_per_frame[4] > 0
        got = h.batch_cone_colors()
        _assert_same(got, _per_frame(h, cl, off))
        for f in (0, 1, 4):
            a, b = int(off[f]), int(off[f + 1])
            assert np.array_equal(got[3][a:b], _oracle_counts(frames[f], cl[a:b])), f


def _blobs(n_blobs, per_blob, seed):
    """n_blobs dense cone-sized blobs 1 m apart in front of the sensor: one cluster each."""
    rng = np.random.default_rng(seed)
    gx, gy = np.meshgrid(np.arange(2.0, 9.5, 1.0), np.arange(-6.0, 6.5, 1.0))
    centres = np.stack([gx.ravel(), gy.ravel()], 1)
    centres = centres[np.hypot(centres[:, 0], centres[:, 1]) < 9.5][:n_blobs]
    assert len(centres) == n_blobs
    out = []
    for cx, cy in centres:
        p = np.empty((per_blob, 4), np.float32)
        p[:, 0] = cx + rng.uniform(-0.1, 0.1, per_blob)
        p[:, 1] = cy + rng.uniform(-0.1, 0.1, per_blob)
        p[:, 2] = rng.uniform(-0.3, 0.0, per_blob)
        p[:, 3] = rng.uniform(0, 255, per_blob)
        out.append(p)
    cloud = np.concatenate(out)
    return cloud[rng.permutation(len(cloud))]


def test_batch_colors_many_clusters_in_one_frame_and_crop_buffer_growth():
    cfg = scans.config(2)
    dense = _blobs(90, 900, 1)                        # 90 clusters in one frame, 81 000 crop points
    other = _bright(scans.generate(cfg, 1, base_seed=60))[0]
    frames = [other, dense]
    with _handle(sum(len(f) for f in frames), 2) as h:   # a fresh handle: the crop buffer starts at 65 536 points
        _, off, cl = h.detect_batch([PointCloud2.from_xyzi(f) for f in frames], cfg.detect, None)
        assert off[2] - off[1] == 90
        got = h.batch_cone_colors()
        assert int(got[3].sum()) > 65536
        assert np.array_equal(got[3][off[1]:], _oracle_counts(dense, cl[off[1]:]))
        assert np.array_equal(got[3][:off[1]], _oracle_counts(other, cl[:off[1]]))
        _assert_same(got, _per_frame(h, cl, off))
        _assert_cpu_chain(tuple(x[off[1]:] for x in got), dense, cl[off[1]:])


def test_batch_colors_extension_values():
    cfg = scans.config(2)
    frames = _bright(scans.generate(cfg, 4, base_seed=70))
    with _handle(4 * cfg.points_per_frame, 4) as h:
        _, off, cl = h.detect_batch([PointCloud2.from_xyzi(f) for f in frames], cfg.detect, cfg.ground)
        for ext in (0.0, -0.05, 1000.0):
            got = h.batch_cone_colors(extension_length=ext)
            _assert_same(got, _per_frame(h, cl, off, ext))
            if ext == 1000.0:               # every box lies far outside the scan
                assert np.all(got[2] == api.CONE_EMPTY) and np.all(got[0] == api.COLOR_NO_ANSWER)
                assert not got[3].any()
            else:
                assert got[3].sum() > 0
        for ext, width in ((float("nan"), 0.228), (float("inf"), 0.228), (-float("inf"), 0.228),
                           (0.05, 0.0), (0.05, -0.228), (0.05, float("nan")), (0.05, float("inf"))):
            with pytest.raises(api.ConesGpuError) as e:
                h.batch_cone_colors(cone_width=width, extension_length=ext)
            assert e.value.status == api.CP_E_PARAM


def _raw_colors(h, K, cap=None, colors=True):
    out = np.zeros(K, np.uint8), np.zeros((K, 3), np.float32), np.zeros(K, np.uint32), np.zeros(K, np.uint32)
    st = h.lib.cp_batch_cone_colors(h._h, C.c_float(0.228), C.c_double(EXT), out[0].ctypes.data if colors else None,
                                    out[1].ctypes.data, out[2].ctypes.data, out[3].ctypes.data,
                                    K if cap is None else cap)
    return st, out


def _results_bytes(h):
    ctr, off, cl = h.results()
    return ctr.tobytes() + off.tobytes() + cl.tobytes()


@pytest.mark.parametrize("case", ["back_half_retry", "graph_replay", "single_launch", "single_off", "back_mode_3"])
def test_batch_colors_come_from_the_final_results(case):
    if case == "back_half_retry":
        cfg = scans.config(4)
        frames = [_bright(scans.generate(cfg, 1, base_seed=0))[0]]     # too dense for the shared-memory back half
        g, kw = None, {}
    else:
        cfg = scans.config(2)
        frames = list(_bright(scans.generate(cfg, 1 if case.startswith("single") else 4, base_seed=80)))
        g = cfg.ground
        kw = {"back_mode": 3} if case == "back_mode_3" else {}
        if case == "single_off":
            kw["env"] = {"CONESGPU_SINGLE": "0"}
    with _handle(sum(len(f) for f in frames), len(frames), **kw) as h:
        msgs = [PointCloud2.from_xyzi(f) for f in frames]
        if case.startswith("single"):
            cl, _ = h.detect(msgs[0], cfg.detect, g)
            h.n_frames = 1
            if case == "single_launch":
                assert h.last_launch_count() == 1
        else:
            h.set_host_input(msgs)
            for _ in range(3 if case == "graph_replay" else 1):   # the third identical run replays a graph
                h.run(cfg.detect, g)
            # straight to the colour call: it must wait for (and, here, redo) the back half itself
            st, raw = _raw_colors(h, 1 << 16)
            assert st == api.CP_OK
        before = _results_bytes(h)
        _, off, cl2 = h.results()
        if case.startswith("single"):
            assert np.array_equal(cl.view(np.uint32), cl2.view(np.uint32))
        cl = cl2
        got = h.batch_cone_colors()
        assert len(cl) > 0
        if not case.startswith("single"):
            assert all(np.array_equal(a, b[:len(cl)]) for a, b in zip(got, raw))
        assert _results_bytes(h) == before
        _assert_same(got, _per_frame(h, cl, off))
        assert _results_bytes(h) == before
        if case == "back_half_retry":
            exp, _, _ = O.detect(O.view_of_xyzi(frames[0]), cfg.detect, None, O.CANONICAL)
            assert np.array_equal(cl.view(np.uint32), exp.view(np.uint32))


def test_batch_colors_errors_and_launch_count():
    cfg = scans.config(3)
    frames = _bright(scans.generate(cfg, 64, base_seed=90))
    with api.ConesGpu(max_points=64 * cfg.points_per_frame, max_frames=64) as h:
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames[:2]])
        h.run(cfg.detect, cfg.ground)
        h.sync()
        assert _raw_colors(h, 64)[0] == api.CP_E_STATE      # no colour net loaded
    with _handle(64 * cfg.points_per_frame, 64) as h:
        assert _raw_colors(h, 64)[0] == api.CP_E_STATE      # no run
        msgs = [PointCloud2.from_xyzi(f) for f in frames]
        h.set_host_input(msgs[:2])
        h.run(cfg.detect, cfg.ground)
        h.set_host_input(msgs[2:4])                          # input staged again since the run
        assert _raw_colors(h, 64)[0] == api.CP_E_STATE
        h.run(cfg.detect, cfg.ground)
        _, _, cl = h.results()
        K = len(cl)
        assert K > 0
        assert _raw_colors(h, K, cap=K - 1)[0] == api.CP_E_CAPACITY
        assert _raw_colors(h, K, colors=False)[0] == api.CP_E_PARAM
        assert _raw_colors(h, K)[0] == api.CP_OK
        launches = {}
        for n in (64, 8):
            h.set_host_input(msgs[:n])
            h.run(cfg.detect, cfg.ground)
            h.batch_cone_colors()                            # grows the buffers for this size
            h.batch_cone_colors()
            launches[n] = h.last_launch_count()
        assert launches[8] == launches[64] > 0, launches


def test_batch_colors_full_config3_batch():
    import torch
    cfg = scans.config(3)
    F = 512
    frames = _bright(scans.generate(cfg, F, base_seed=100))
    dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()
    with _handle(F * cfg.points_per_frame, F) as h:
        h.set_device_input(dev.data_ptr(), np.full(F, cfg.points_per_frame, np.uint32), keep=dev)
        h.run(cfg.detect, cfg.ground)
        _, off, cl = h.results()
        got = h.batch_cone_colors()
        assert len(cl) > 10 * F
        _assert_same(got, _per_frame(h, cl, off))
