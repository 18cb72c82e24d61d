"""What the cone-detection node publishes, over frame sequences on the device (cp_batch_track), bit for bit.

The oracle is tests/util.TrackerReference (src/cone_detection.cpp:276-340 restated), driven frame by frame with the
run's records.  Its colour callback receives centres; the wrapper here maps them back to the frame's records by their
exact float bits and applies the service's response rules (a bad crop fails the call, empty crops are skipped) to
per-record answers: the device's (cp_batch_cone_colors) or, for a few frames, the CPU chain.  Compared: x / y as
uint32, order, colour, cluster and the cloud offsets."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200 import tflite_model as T
from cones_perception_b200.pointcloud2 import PointCloud2, PointField
from oracle import dam_net_ref as D
from oracle import oracle as O
from tests.util import TrackerReference

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXT, WIDTH = 0.05, 0.228
BAD = api.CONE_BAD_INDEX | api.CONE_BAD_INTENSITY


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


def _ext(x, y, ext=EXT):
    """The extended centre exactly as TrackerReference computes it."""
    f32, f64 = np.float32, np.float64
    px, py = f32(x), f32(y)
    with np.errstate(all="ignore"):
        ln = TrackerReference.dist((px, py, f32(0)), (0, 0, 0))
        return f32(f64(px) + f64(f32(px / ln)) * ext), f32(f64(py) + f64(f32(py / ln)) * ext)


def _key(x, y):
    return (int(np.float32(x).view(np.uint32)), int(np.float32(y).view(np.uint32)))


class Answers:
    """color_fn for TrackerReference: per-record answers of frame f, response rules of ConeDetector::gpu_colors."""

    def __init__(self, colors, flags, ext=EXT):
        self.colors, self.flags, self.ext = colors, flags, ext
        self.asked = {}   # frame's first record -> keys of the centres the node asked colours for

    def set_frame(self, recs, base):
        self.base = base
        self.asked[base] = set()
        self.index = {}
        for i, r in enumerate(recs):
            self.index.setdefault(_key(*_ext(r["x"], r["y"], self.ext)), base + i)

    def __call__(self, centres):
        self.asked[self.base] |= {_key(p[0], p[1]) for p in centres}
        ks = [self.index[_key(p[0], p[1])] for p in centres]
        if any(int(self.flags[k]) & BAD for k in ks):
            return []
        return [int(self.colors[k]) if self.colors[k] < 4 else 0 for k in ks if not self.flags[k] & api.CONE_EMPTY]


def reference(clusters, off, seqs, params, answers=None, slots=None):
    """TrackerReference per sequence; slots (dict, sequence index -> reference) carries state across calls.
    Returns (cones, cloud_offsets) in the device's layout."""
    F = len(off) - 1
    slots = {} if slots is None else slots
    cones, coff = [], [0]
    frame_clouds = [None] * F
    for s in range(len(seqs) - 1):
        if s not in slots:
            slots[s] = TrackerReference(bool(params.classify_colors), bool(params.use_points_buffer),
                                        params.cones_matching_dist_theshold, params.cone_position_extension_length,
                                        color_fn=answers)
        t = slots[s]
        t.color_fn = answers
        for f in range(seqs[s], seqs[s + 1]):
            recs = clusters[off[f]:off[f + 1]]
            if answers is not None:
                answers.set_frame(recs, int(off[f]))
            frame_clouds[f] = t.update([(r["x"], r["y"]) for r in recs])
    for f in range(F):
        index = {}
        for i, r in enumerate(clusters[off[f]:off[f + 1]]):
            index.setdefault(_key(*_ext(r["x"], r["y"], params.cone_position_extension_length)), int(off[f]) + i)
        for c in range(4):
            for p in frame_clouds[f][c]:
                cones.append((p[0], p[1], index[_key(p[0], p[1])], c))
            coff.append(len(cones))
    out = np.zeros(len(cones), api.TRACKED_CONE_DTYPE)
    for i, c in enumerate(cones):
        out[i] = c
    return out, np.array(coff, np.uint32)


def assert_same(got, exp):
    cones, coff = got
    ec, eo = exp
    assert np.array_equal(coff, eo), (coff, eo)
    for a in ("x", "y"):   # NaN (a centroid at the origin) compares as NaN: its bits are the platform's default NaN
        g, e = cones[a].copy(), ec[a].copy()
        assert np.array_equal(np.isnan(g), np.isnan(e))
        g[np.isnan(g)] = 0
        e[np.isnan(e)] = 0
        assert np.array_equal(g.view(np.uint32), e.view(np.uint32)), a
    assert np.array_equal(cones["color"], ec["color"])
    # a record whose extended centre repeats another's in the same frame maps to the first: compare the centres
    assert np.array_equal(cones["cluster"], ec["cluster"]) or _same_centres(cones, ec)


def _same_centres(a, b):
    return np.array_equal(a["x"].view(np.uint32), b["x"].view(np.uint32)) or bool(np.isnan(a["x"]).any())


def _seqs(n_frames, seq_offsets):
    return list(seq_offsets) if seq_offsets is not None else [0, n_frames]


def _two_scenes(cfg, seed):
    """16 frames: 8 of a scene, then 8 of it moved 0.7 m sideways, so that the points buffer drops cones at the cut."""
    a = scans.generate(cfg, 16, base_seed=seed)
    a[8:, :, 1] += np.float32(0.7)
    return a


def _run(h, frames, cfg, g="cfg"):
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    _, off, cl = h.detect_batch(msgs, cfg.detect, cfg.ground if g == "cfg" else g)
    return off, cl


# ---- CPU ------------------------------------------------------------------------------------------------------
def test_track_struct_layout_matches_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "conesgpu.h"\n#include <stddef.h>\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu\\n", sizeof(cp_track_params), sizeof(cp_tracked_cone),'
                   ' offsetof(cp_track_params, cones_matching_dist_theshold), offsetof(cp_track_params, cone_width),'
                   ' offsetof(cp_tracked_cone, color));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(api.CTrackParams), C.sizeof(api.CTrackedCone), api.CTrackParams.cones_matching_dist_theshold.offset,
                   api.CTrackParams.cone_width.offset, api.CTrackedCone.color.offset]
    assert C.sizeof(api.CTrackedCone) == api.TRACKED_CONE_DTYPE.itemsize == 16


# ---- GPU: runs --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("buffer", [False, True])
def test_gate_without_colours(buffer):
    cfg = scans.config(2)
    frames = _two_scenes(cfg, 210)
    with _handle(16 * cfg.points_per_frame, 16, net=False) as h:
        off, cl = _run(h, frames, cfg)
        p = api.track_params(False, buffer)
        got = h.batch_track(p)
        exp = reference(cl, off, [0, 16], p)
        assert_same(got, exp)
        assert len(got[0]) > 0 and got[1][4] == 0          # the first frame publishes nothing
        if buffer:
            assert len(got[0]) < len(cl) - (off[1] - off[0])  # some cones fail the points buffer


def _colour_case(h, frames, cfg, p, seq_offsets=None):
    off, cl = _run(h, frames, cfg)
    colors, _, flags, _ = h.batch_cone_colors(WIDTH, p.cone_position_extension_length)
    got = h.batch_track(p, seq_offsets)
    ans = Answers(colors, flags, p.cone_position_extension_length)
    exp = reference(cl, off, _seqs(len(frames), seq_offsets), p, ans)
    assert_same(got, exp)
    return off, cl, got, colors, flags, ans


@pytest.mark.gpu
@pytest.mark.parametrize("buffer", [False, True])
def test_colours_with_the_device_net(buffer):
    cfg = scans.config(2)
    frames = _bright(_two_scenes(cfg, 220))
    with _handle(16 * cfg.points_per_frame, 16) as h:
        p = api.track_params(True, buffer)
        off, cl, (cones, coff), colors, flags, ans = _colour_case(h, frames, cfg, p)
        K = len(cl)
        published = np.zeros(K, bool)
        published[cones["cluster"]] = True
        first = np.zeros(K, bool)
        first[off[0]:off[1]] = True
        if buffer:   # without the points buffer every cone passes once the previous frame had one
            assert (~published & ~first).any(), "no gated-out cone"
        # fresh: the node asked the service for this cone's colour; carried: published in a colour cloud unasked
        fresh = carried = 0
        frame_of = np.searchsorted(off, cones["cluster"], side="right") - 1
        for c, f in zip(cones, frame_of):
            if c["color"] == 0:
                continue
            if _key(c["x"], c["y"]) in ans.asked[int(off[f])]:
                fresh += 1
            else:
                carried += 1
        assert fresh > 0 and carried > 0, (fresh, carried)
        # the CPU chain on two frames gives the same answers the device used
        g = T.load(_model())
        for f in (1, 15):
            pts = O.points32(frames[f])
            for k in range(off[f], off[f + 1]):
                if flags[k] & (api.CONE_AMBIGUOUS | api.CONE_LOW_CONFIDENCE):
                    continue
                crop = O.reconstruct_cone(pts, *_ext(cl[k]["x"], cl[k]["y"]))
                if len(crop) == 0:
                    assert flags[k] & api.CONE_EMPTY
                    continue
                img, fl = O.to_image(np.stack([crop["x"], crop["y"], crop["z"], crop["intensity"]], 1))
                if fl == 0:
                    assert int(colors[k]) == D.decide(D.forward(g, img)[0]), k


def _ragged_frames():
    cfg = scans.config(1)
    src = _bright(scans.generate(cfg, 4, base_seed=230))
    far = src[2].copy()
    far[:, :2] *= 100.0
    return cfg, [src[0], src[1][:17001], np.zeros((0, 4), np.float32), far, src[2], src[3]]


def _layout_msg(frame, step, offs):
    n = len(frame)
    raw = np.zeros((n, step), np.uint8)
    for k, o in enumerate(offs):
        raw[:, o:o + 4] = frame[:, k].copy().view(np.uint8).reshape(n, 4)
    return PointCloud2(data=raw.reshape(-1), width=n, height=1, point_step=step,
                       fields=[PointField(nm, o) for nm, o in zip(("x", "y", "z", "intensity"), offs)])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["device", "pcl32", "odd"])
def test_several_sequences_every_input_layout(layout):
    cfg, frames = _ragged_frames()
    total = sum(len(f) for f in frames)
    # sequences: frames 0-1, an empty one, frame 2 alone (empty frame), frames 3-5 (3 has no cluster)
    seq = np.array([0, 2, 2, 3, 6], np.uint32)
    with _handle(total, len(frames), max_point_step=32) as h:
        if layout == "device":
            import torch
            dev = torch.from_numpy(np.ascontiguousarray(np.concatenate(frames))).cuda()
            h.set_device_input(dev.data_ptr(), np.array([len(f) for f in frames], np.uint32), keep=dev)
        elif layout == "pcl32":
            h.set_host_input([_layout_msg(f, 32, (0, 4, 8, 16)) for f in frames])
        else:
            h.set_host_input([_layout_msg(f, 23, (1, 5, 9, 14)) for f in frames])
        h.run(cfg.detect, cfg.ground)
        _, off, cl = h.results()
        assert np.diff(off)[2] == 0 and np.diff(off)[3] == 0 and np.diff(off)[4] > 0
        colors, _, flags, _ = h.batch_cone_colors()
        for buffer in (False, True):
            h.track_reset()
            h.run(cfg.detect, cfg.ground)
            p = api.track_params(True, buffer)
            got = h.batch_track(p, seq)
            assert_same(got, reference(cl, off, seq, p, Answers(colors, flags)))
            assert got[1][4 * 5] == got[1][4 * 4]            # frame 4 follows a frame without clusters


@pytest.mark.gpu
@pytest.mark.parametrize("classify", [False, True])
def test_continuity_across_calls(classify):
    cfg = scans.config(2)
    frames = _bright(scans.generate(cfg, 24, base_seed=240))
    p = api.track_params(classify, True)
    n = cfg.points_per_frame
    with _handle(24 * n, 24) as h:
        msgs = [PointCloud2.from_xyzi(f) for f in frames]
        _, off, cl = h.detect_batch(msgs, cfg.detect, cfg.ground)
        one = h.batch_track(p)
        h.track_reset()
        parts = []
        for b in range(3):
            _, o, _ = h.detect_batch(msgs[8 * b:8 * b + 8], cfg.detect, cfg.ground)
            c, co = h.batch_track(p)
            c["cluster"] += off[8 * b]
            parts.append((c, co[:-1] + (int(sum(len(x[0]) for x in parts)))))
        three = np.concatenate([x[0] for x in parts]), np.concatenate([x[1] for x in parts] + [[len(one[0])]])
        assert_same(three, one)
        h.track_reset()
        singles = []
        for f in range(24):
            cl1, _ = h.detect(msgs[f], cfg.detect, cfg.ground)
            c, co = h.batch_track(p)
            if f == 0:
                assert len(c) == 0
            c["cluster"] += off[f]
            singles.append(c)
        assert_same((np.concatenate(singles), one[1]), one)
        h.track_reset()
        h.detect_batch(msgs[5:6], cfg.detect, cfg.ground)
        c, co = h.batch_track(p)
        assert len(c) == 0 and not co.any()                   # after a reset the first frame publishes nothing


# ---- GPU: constructed records (cp_debug_track) ----------------------------------------------------------------
def _recs(xy):
    r = np.zeros(len(xy), api.CLUSTER_DTYPE)
    if len(xy):
        r["x"], r["y"] = np.asarray(xy, np.float32).T
    r["size"] = 3
    return r


def _debug(h, p, frames_xy, colors=None, flags=None, seq=None, slots=None):
    recs = _recs([xy for fr in frames_xy for xy in fr])
    off = np.concatenate([[0], np.cumsum([len(fr) for fr in frames_xy])]).astype(np.uint32)
    got = h.debug_track(p, recs, off, colors, flags, seq)
    ans = Answers(colors, flags, p.cone_position_extension_length) if colors is not None else None
    exp = reference(recs, off, _seqs(len(frames_xy), seq), p, ans, slots)
    assert_same(got, exp)
    return got


def _threshold_pairs():
    """(p, q) along x at distances whose float32 sits just below, at and above 0.5 (searched in float/double)."""
    base = np.float32(3.0)
    pairs = []
    q = np.float32(3.5)
    ref = TrackerReference
    for step in range(-6, 7):
        qq = np.float32(q + np.float32(step) * np.spacing(q))
        pairs.append(((float(base), 0.0), (float(qq), 0.0)))
    # a diagonal pair whose double distance rounds onto 0.5 in float
    for k in range(200):
        y = np.float32(0.3 + k * 1e-9)
        x = np.float32(np.sqrt(0.25 - np.float64(y) ** 2))
        if ref.dist((x, y, 0), (0, 0, 0)) == np.float32(0.5):
            pairs.append(((5.0, 5.0), (float(np.float32(5.0) + x), float(np.float32(5.0) + y))))
    return pairs


@pytest.mark.gpu
def test_debug_threshold_origin_and_big_frames():
    with _handle(1 << 16, 64, net=False) as h:
        for buffer in (False, True):
            p = api.track_params(False, buffer, ext=0.0)
            pairs = _threshold_pairs()
            d = [TrackerReference.dist((np.float32(a[0]), np.float32(a[1]), 0), (np.float32(b[0]), np.float32(b[1]), 0))
                 for a, b in pairs]
            assert any(x < 0.5 for x in d) and any(x == np.float32(0.5) for x in d) and any(x > 0.5 for x in d)
            for a, b in pairs:
                h.track_reset()
                _debug(h, p, [[a], [b]])
            h.track_reset()
            _debug(h, api.track_params(False, buffer), [[(0.0, 0.0), (1.0, 1.0)], [(0.0, 0.0), (1.0, 1.02)]])
            rng = np.random.default_rng(1)
            blob = [(float(2 + rng.uniform(0, 0.2)), float(rng.uniform(0, 0.2))) for _ in range(2000)]
            h.track_reset()
            got = _debug(h, api.track_params(False, buffer), [blob, blob[::-1]])
            assert len(got[0]) == 2000


@pytest.mark.gpu
def test_debug_response_rules():
    with _handle(1 << 16, 64, net=False) as h:
        p = api.track_params(True, True)
        xy = [(3.0 + i, 0.5 * i) for i in range(40)]
        frames = [xy, [(x + 0.01, y) for x, y in xy], [(x + 0.02, y) for x, y in xy]]
        K = 120
        colors = np.array([(i % 3) + 1 for i in range(K)], np.uint8)
        flags = np.zeros(K, np.uint32)
        flags[45] = flags[50] = api.CONE_EMPTY                    # skipped: later colours move up
        colors[45] = colors[50] = 255
        got = _debug(h, p, frames, colors, flags)
        assert len(got[0]) > 0
        h.track_reset()
        flags2 = flags.copy()
        flags2[47] = api.CONE_BAD_INTENSITY                      # the whole call fails: every need colour is 0
        colors[47] = 255
        got = _debug(h, p, frames, colors, flags2)
        c1 = got[0][got[1][4]:got[1][8]]
        assert len(c1) == 40 and np.all(c1["color"] == 0)


@pytest.mark.gpu
def test_debug_long_sequence_and_many_sequences():
    rng = np.random.default_rng(3)
    F = 4096
    frames = [[(float(5 + rng.normal(0, 0.3)), float(rng.normal(0, 2))) for _ in range(rng.integers(0, 6))]
              for _ in range(F)]
    K = sum(len(f) for f in frames)
    colors = rng.integers(0, 4, K).astype(np.uint8)
    flags = np.where(rng.random(K) < 0.1, api.CONE_EMPTY, 0).astype(np.uint32)
    colors[flags != 0] = 255
    with _handle(1 << 16, 64, net=False) as h:
        for buffer in (False, True):
            h.track_reset()
            _debug(h, api.track_params(True, buffer, match=0.7), frames, colors, flags)
        # max_frames sequences of 64 frames, in two calls: state continues per slot
        seq = np.arange(0, F + 1, 64, dtype=np.uint32)
        h.track_reset()
        slots = {}
        p = api.track_params(True, True, match=0.7)
        for half in range(2):
            part = frames[half * 2048:(half + 1) * 2048]
            a = sum(len(f) for f in frames[:half * 2048])
            b = a + sum(len(f) for f in part)
            _debug(h, p, part, colors[a:b], flags[a:b], np.arange(0, 2049, 32, dtype=np.uint32), slots)


# ---- GPU: errors and invariance --------------------------------------------------------------------------------
def _raw_track(h, p, seq=None, n_seqs=None, cap=1 << 16, out=True, coff=True, F=None):
    F = h.n_frames if F is None else F
    o = np.zeros(max(cap, 1), api.TRACKED_CONE_DTYPE)
    co = np.zeros(4 * F + 1, np.uint32)
    n = C.c_uint64(12345)
    so = np.ascontiguousarray(seq, np.uint32) if seq is not None else None
    st = h.lib.cp_batch_track(h._h, C.byref(p), so.ctypes.data if so is not None else None,
                              (len(so) - 1 if so is not None else 1) if n_seqs is None else n_seqs,
                              o.ctypes.data if out else None, co.ctypes.data if coff else None, cap, C.byref(n))
    return st, o[:n.value], co, n.value


@pytest.mark.gpu
def test_errors_leave_the_state_alone():
    cfg = scans.config(3)
    frames = _bright(scans.generate(cfg, 8, base_seed=250))
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    p = api.track_params(True, True)
    with _handle(8 * cfg.points_per_frame, 8, net=False) as h:
        h.n_frames = 4
        assert _raw_track(h, api.track_params())[0] == api.CP_E_STATE            # no run
        h.detect_batch(msgs[:4], cfg.detect, cfg.ground)
        assert _raw_track(h, p)[0] == api.CP_E_STATE                             # no net
    with _handle(8 * cfg.points_per_frame, 8) as h, _handle(8 * cfg.points_per_frame, 8) as ref:
        for x in (h, ref):
            x.detect_batch(msgs[:4], cfg.detect, cfg.ground)
        exp1 = ref.batch_track(p)
        _, off, cl = h.results()
        K = len(cl)
        bad = [api.track_params(True, True, match=float("nan")), api.track_params(True, True, ext=float("inf")),
               api.track_params(True, True, cone_width=0.0), api.track_params(True, True, cone_width=float("nan"))]
        for q in bad:
            assert _raw_track(h, q)[0] == api.CP_E_PARAM
        assert _raw_track(h, api.track_params(False, True, cone_width=0.0))[0] == api.CP_OK   # width unused
        h.track_reset()
        h.run(cfg.detect, cfg.ground)
        for seq, n in (([0, 3, 2, 4], None), ([1, 4], None), ([0, 3], None), (None, 2), ([0, 4], 0),
                       (list(range(0, 5)) + [4] * 5, None)):
            assert _raw_track(h, p, seq, n)[0] == api.CP_E_PARAM, (seq, n)
        assert _raw_track(h, p, coff=False)[0] == api.CP_E_PARAM
        st, _, _, n = _raw_track(h, p, cap=0)
        assert st == api.CP_E_CAPACITY and n == len(exp1[0]) > 0
        assert _raw_track(h, p, out=False)[0] == api.CP_E_PARAM
        st, o, co, n = _raw_track(h, p, cap=K)
        assert st == api.CP_OK
        assert_same((o, co), exp1)
        assert _raw_track(h, p)[0] == api.CP_E_STATE                             # already tracked
        for x in (h, ref):
            x.set_host_input(msgs[4:])
        assert _raw_track(h, p)[0] == api.CP_E_STATE                             # staged since the run
        for x in (h, ref):
            x.run(cfg.detect, cfg.ground)
        assert_same(h.batch_track(p), ref.batch_track(p))


@pytest.mark.gpu
def test_launch_count_and_results_untouched():
    cfg = scans.config(3)
    frames = _bright(scans.generate(cfg, 64, base_seed=260))
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    with _handle(64 * cfg.points_per_frame, 64) as h:
        for classify in (False, True):
            launches = {}
            for n in (64, 8):
                h.detect_batch(msgs[:n], cfg.detect, cfg.ground)
                h.batch_track(api.track_params(classify, True), [0, n // 2, n])
                h.run(cfg.detect, cfg.ground)
                ctr, off, cl = h.results()
                before = ctr.tobytes() + off.tobytes() + cl.tobytes()
                d_cl, d_off, _ = h.device_results()
                dev_before = _dev_bytes(d_off, (n + 1) * 4), _dev_bytes(d_cl, len(cl) * 16)
                h.batch_track(api.track_params(classify, True), [0, n // 2, n])
                launches[n] = h.last_launch_count()
                ctr, off, cl = h.results()
                assert ctr.tobytes() + off.tobytes() + cl.tobytes() == before
                assert (_dev_bytes(d_off, (n + 1) * 4), _dev_bytes(d_cl, len(cl) * 16)) == dev_before
            assert launches[8] == launches[64] > 0, launches


class _DevView:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def _dev_bytes(ptr, nbytes):
    """Bytes of device memory the library owns (zero-copy view through __cuda_array_interface__)."""
    import torch
    torch.cuda.synchronize()
    return torch.as_tensor(_DevView(ptr, nbytes), device="cuda").cpu().numpy().tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["back_half_retry", "graph_replay"])
def test_after_retry_and_graph_replay(case):
    if case == "back_half_retry":
        cfg = scans.config(4)
        frames = list(_bright(scans.generate(cfg, 2, base_seed=270)))
        g = None
    else:
        cfg = scans.config(2)
        frames = list(_bright(scans.generate(cfg, 4, base_seed=280)))
        g = cfg.ground
    with _handle(sum(len(f) for f in frames), len(frames)) as h:
        h.set_host_input([PointCloud2.from_xyzi(f) for f in frames])
        for _ in range(3 if case == "graph_replay" else 1):
            h.run(cfg.detect, g)
        p = api.track_params(True, True)
        st, o, co, n = _raw_track(h, p)                      # straight after the run: waits for the final records
        assert st == api.CP_OK
        _, off, cl = h.results()
        colors, _, flags, _ = h.batch_cone_colors()
        assert_same((o, co), reference(cl, off, [0, len(frames)], p, Answers(colors, flags)))
        if case == "back_half_retry":
            exp, _, _ = O.detect(O.view_of_xyzi(frames[0]), cfg.detect, None, O.CANONICAL)
            assert np.array_equal(cl[off[0]:off[1]].view(np.uint32), exp.view(np.uint32))


@pytest.mark.gpu
def test_full_config3_batch_as_8_sequences():
    import torch
    cfg = scans.config(3)
    F = 512
    frames = _bright(scans.generate(cfg, F, base_seed=290))
    dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()
    seq = np.arange(0, F + 1, 64, dtype=np.uint32)
    with _handle(F * cfg.points_per_frame, F) as h:
        h.set_device_input(dev.data_ptr(), np.full(F, cfg.points_per_frame, np.uint32), keep=dev)
        for classify in (False, True):
            h.track_reset()
            h.run(cfg.detect, cfg.ground)
            _, off, cl = h.results()
            assert len(cl) > 10 * F
            colors, _, flags, _ = h.batch_cone_colors()
            p = api.track_params(classify, True)
            got = h.batch_track(p, seq)
            assert_same(got, reference(cl, off, seq, p, Answers(colors, flags) if classify else None))


# ---- GPU: the C++ node layer -----------------------------------------------------------------------------------
def _host_lib():
    from cones_perception_b200.build import HOST_LIB
    lib = C.CDLL(HOST_LIB)
    lib.ch_last_error.restype = C.c_char_p
    lib.ch_detector_create.restype = C.c_void_p
    lib.ch_detector_create.argtypes = [C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.ch_detector_create_replay.restype = C.c_void_p
    lib.ch_detector_create_replay.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.ch_detector_destroy.argtypes = [C.c_void_p]
    lib.ch_detector_load_color_model.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    lib.ch_detector_publish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                        C.c_uint64, C.POINTER(C.c_uint64)]
    return lib


def _publish(lib, det, frames, replay):
    xyzi = np.ascontiguousarray(np.concatenate(frames), np.float32)
    n = np.array([len(f) for f in frames], np.uint32)
    out = np.zeros(64 << 20, np.uint8)
    used = C.c_uint64()
    rc = lib.ch_detector_publish(det, xyzi.ctypes.data, n.ctypes.data, len(frames), 1, int(replay), out.ctypes.data,
                                 out.nbytes, C.byref(used))
    assert rc == 0, lib.ch_last_error()
    return out[:used.value].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("classify", [False, True])
@pytest.mark.parametrize("buffer", [False, True])
def test_cpp_replay_publishes_what_cloud_handler_publishes(classify, buffer):
    from cones_perception_b200.params import to_c_detect
    lib = _host_lib()
    cfg = scans.config(2)
    frames = list(_bright(scans.generate(cfg, 10, base_seed=300)))
    cd = to_c_detect(cfg.detect)
    model = _model()
    buf = (C.c_uint8 * len(model)).from_buffer_copy(model)
    per_msg = lib.ch_detector_create(cfg.points_per_frame, 0, C.byref(cd), int(classify), int(buffer), 1)
    rep = lib.ch_detector_create_replay(4 * cfg.points_per_frame, 4, 0, C.byref(cd), int(classify), int(buffer), 1)
    try:
        assert per_msg and rep, lib.ch_last_error()
        if classify:
            for det in (per_msg, rep):
                assert lib.ch_detector_load_color_model(det, buf, len(model)) == 0, lib.ch_last_error()
        exp = _publish(lib, per_msg, frames, False)
        got = _publish(lib, rep, frames, True)               # three device batches: 4 + 4 + 2 messages
        assert got == exp
        xyzi = np.ascontiguousarray(frames[0])
        n = np.array([len(xyzi)], np.uint32)
        used = C.c_uint64()
        out = np.zeros(1 << 20, np.uint8)
        # the per-message entry on the replaying object is refused: the two would share one node state
        assert lib.ch_detector_publish(rep, xyzi.ctypes.data, n.ctypes.data, 1, 1, 0, out.ctypes.data, out.nbytes,
                                       C.byref(used)) == 4
    finally:
        lib.ch_detector_destroy(per_msg)
        lib.ch_detector_destroy(rep)
