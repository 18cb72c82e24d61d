"""The ground-removal node's groundless_cloud for every frame of a batch (cp_batch_ground_remove), bit for bit.

Every case compares each frame's message (survivors in input order, then the PCL padding points) with
oracle.ground_node on that frame alone, and n_kept and the 17 sector minima (as uint32) with it.  Frames sit back to
back in the output: frame f's message starts at point P_f = sum of the earlier frames' N."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200.params import GroundParams, to_c_ground
from cones_perception_b200.pointcloud2 import PointCloud2
from oracle import oracle as O
from tests.test_gpu_parity import _msg_with_layout
from tests.test_oracle import _outside_sector_16

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
G = GroundParams()
FIELDS = ("x", "y", "z", "pad", "intensity", "c1", "c2", "c3")
TILE = 2048


def _expect(views):
    """Per frame: (message bytes, kept, low17 as uint32) from the oracle's ground node."""
    out = []
    for v in views:
        if v.width * v.height == 0:   # no message body; the minima keep their initial value
            out.append((b"", 0, np.full(17, G.default_lowest_point, np.float32).view(np.uint32)))
            continue
        e, kept, low, _ = O.ground_node(v, G)
        b = np.stack([e[n] for n in FIELDS], 1).astype(np.float32).tobytes() if len(e) else b""
        out.append((b, kept, low.view(np.uint32).copy()))
    return out


def _check(got, kept, low, exp):
    """got: the batch output as bytes (or [sum N, 8] float32)."""
    raw = got if isinstance(got, bytes) else np.ascontiguousarray(got).tobytes()
    assert len(raw) == sum(len(e[0]) for e in exp)
    at = 0
    for f, (b, k, lo) in enumerate(exp):
        assert raw[at:at + len(b)] == b, f"frame {f}: message differs"
        assert int(kept[f]) == k, (f, int(kept[f]), k)
        assert np.array_equal(low[f].view(np.uint32), lo), f"frame {f}: sector minima differ"
        at += len(b)


class _DevView:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def _dev_bytes(ptr, nbytes):
    import torch
    torch.cuda.synchronize()
    if nbytes == 0:
        return b""
    return torch.as_tensor(_DevView(ptr, nbytes), device="cuda").cpu().numpy().tobytes()


def _ragged():
    """An empty frame, a 1-point frame, exactly one tile, one point past a tile, an all-ground frame (G = 0), a
    no-ground frame (G = N, minima at default_lowest_point), the reference node's two golden frames at non-zero
    offsets, and ordinary scans around them."""
    cfg = scans.config(2)
    src = scans.generate(cfg, 3, base_seed=900)
    gold = [_outside_sector_16(scans.generate(cfg, 1, base_seed=s)[0]) for s in (0, 9)]
    flat = src[1][:3000].copy()
    flat[:, 2] = -1.0                                     # every point is its sector's minimum: all ground
    high = src[2][:5000].copy()
    high[:, 2] = np.abs(high[:, 2]) + 0.5                 # nothing below default_lowest_point + 0.1
    frames = [src[0], gold[0], np.zeros((0, 4), np.float32), src[1][:1], src[1][70000:70000 + TILE],
              src[2][90000:90000 + TILE + 1],
              flat, high, gold[1], src[2]]
    return [np.ascontiguousarray(f, np.float32) for f in frames], {"gold": (1, 8), "flat": 6, "high": 7}


def _msgs(frames):
    return [PointCloud2.from_xyzi(f) for f in frames]


def _views(msgs):
    return [O.view_of_msg(m, fake_missing_intensity=False) for m in msgs]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["host", "device"])
def test_ragged_batch_against_oracle_goldens_and_single_frame(path):
    frames, where = _ragged()
    msgs = _msgs(frames)
    exp = _expect(_views(msgs))
    total = sum(len(f) for f in frames)
    with api.ConesGpu(max_points=total, max_frames=len(frames), max_point_step=32) as h:
        if path == "host":
            h.set_host_input(msgs, fake_missing_intensity=False)
        else:
            import torch
            dev = torch.from_numpy(np.ascontiguousarray(np.concatenate(frames))).cuda()
            h.set_device_input(dev.data_ptr(), [len(f) for f in frames], 16, (0, 4, 8, 12), keep=dev)
        out, kept, low = h.batch_ground_remove(G)
        _check(out, kept, low, exp)
        ptr, n = h.ground_device_output()
        assert n == total and _dev_bytes(ptr, 32 * n) == out.tobytes()
        _, dkept, dlow = h.batch_ground_remove(G, host=False)   # device output only
        assert np.array_equal(dkept, kept) and np.array_equal(dlow.view(np.uint32), low.view(np.uint32))
        ptr, n = h.ground_device_output()
        assert _dev_bytes(ptr, 32 * n) == out.tobytes()
    # the regimes the batch is meant to reach
    assert kept[where["flat"]] == 0 and kept[where["high"]] == len(frames[where["high"]])
    assert np.all(low[where["high"]] == np.float32(G.default_lowest_point))
    assert kept[2] == 0 and len(frames[2]) == 0
    # the reference node's goldens, placed inside the batch
    z = np.load(os.path.join(GOLD, "reference_nodes.npz"))
    off = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    for seed, f in zip((0, 9), where["gold"]):
        assert off[f] > 0
        assert hashlib.sha256(frames[f].tobytes()).hexdigest() == str(z[f"ground_seed{seed}_input_sha256"])
        assert int(kept[f]) == int(z[f"ground_seed{seed}_kept"])
        assert hashlib.sha256(out[off[f]:off[f + 1]].tobytes()).hexdigest() == str(z[f"ground_seed{seed}_sha256"])
    # every frame equals cp_ground_remove on that frame alone
    with api.ConesGpu(max_points=max(len(f) for f in frames)) as one:
        for f, m in enumerate(msgs):
            if len(frames[f]) == 0:
                continue
            o1, k1, _ = one.ground_remove(m, G)
            assert k1 == kept[f]
            assert hashlib.sha256(o1.tobytes()).hexdigest() == hashlib.sha256(out[off[f]:off[f + 1]].tobytes()).hexdigest()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["pcl32", "unaligned22", "organised"])
def test_input_layouts_staged_from_the_host(layout):
    cfg = scans.config(1)
    src = scans.generate(cfg, 3, base_seed=910)
    frames = [f[:29_984] for f in src]                    # 16 rows of 1874 points
    if layout == "pcl32":
        msgs = [_msg_with_layout(f, 32, (0, 4, 8, 16)) for f in frames]
    elif layout == "unaligned22":
        msgs = [_msg_with_layout(f, 22, (0, 4, 8, 12)) for f in frames]
    else:
        msgs = [_msg_with_layout(f, 32, (0, 4, 8, 16), True, 16, 64) for f in frames]
        assert msgs[0].height == 16 and msgs[0].row_step > msgs[0].width * 32
    exp = _expect(_views(msgs))
    with api.ConesGpu(max_points=sum(len(f) for f in frames), max_frames=3, max_point_step=32) as h:
        h.set_host_input(msgs, fake_missing_intensity=False)
        out, kept, low = h.batch_ground_remove(G)
    _check(out, kept, low, exp)


@pytest.mark.gpu
def test_uniform_config3_batch_of_64():
    cfg = scans.config(3)
    frames = scans.generate(cfg, 64, base_seed=920)
    msgs = _msgs(frames)
    exp = _expect(_views(msgs))
    with api.ConesGpu(max_points=64 * cfg.points_per_frame, max_frames=64) as h:
        h.set_host_input(msgs, fake_missing_intensity=False)
        out, kept, low = h.batch_ground_remove(G)
    _check(out, kept, low, exp)
    assert 0 < kept.min() and kept.max() < cfg.points_per_frame


@pytest.mark.gpu
def test_two_node_chain_on_the_device():
    """Handle A publishes the groundless clouds on the device; handle B detects on them (ground removal off), as the
    reference's launch wires the two nodes.  Cluster records equal the fused run's and the oracle's."""
    import torch
    cfg = scans.config(3)
    F = 16
    frames = scans.generate(cfg, F, base_seed=930)
    msgs = _msgs(frames)
    n = cfg.points_per_frame
    with api.ConesGpu(max_points=F * n, max_frames=F) as a, \
            api.ConesGpu(max_points=F * n, max_frames=F, max_point_step=32) as b, \
            api.ConesGpu(max_points=F * n, max_frames=F) as fused:
        a.set_host_input(msgs, fake_missing_intensity=False)
        _, kept, _ = a.batch_ground_remove(G, host=False)
        ptr, total = a.ground_device_output()
        assert total == F * n
        b.set_device_input(ptr, [n] * F, 32, (0, 4, 8, 16))
        b.run(cfg.detect, None)
        cctr, coff, ccl = b.results()
        fused.set_host_input(msgs)
        fused.run(cfg.detect, G)
        fctr, foff, fcl = fused.results()
    torch.cuda.synchronize()
    assert np.array_equal(coff, foff) and np.array_equal(ccl.view(np.uint32), fcl.view(np.uint32))
    for k in ("n_voxels", "n_components", "n_clusters", "key_bits"):
        assert np.array_equal(cctr[k], fctr[k]), k
    # n_ground_kept differs by wiring: the detection node of the chain removes no ground, so it counts all N points
    # of the groundless message; the fused path counts the G survivors.  n_cropped differs only if the padding
    # point (0, 0, 0) passes the crop: the chain crops its N - G copies one by one, while the fused path models
    # them as one record.
    assert np.all(cctr["n_ground_kept"] == n) and np.array_equal(fctr["n_ground_kept"], kept)
    assert cfg.detect.distance_treshold_min > 0                     # here it does not (distance 0 < the minimum)
    assert np.array_equal(cctr["n_cropped"], fctr["n_cropped"])
    for f in range(0, F, 5):
        e, _, _ = O.detect(O.view_of_xyzi(frames[f]), cfg.detect, G, O.CANONICAL)
        assert np.array_equal(ccl[coff[f]:coff[f + 1]].view(np.uint32), e.view(np.uint32))


def _raw(h, g, out, cap, kept=None, low=None):
    return h.lib.cp_batch_ground_remove(h._h, C.byref(to_c_ground(g)) if g is not None else None,
                                        out.ctypes.data if out is not None else None, cap,
                                        kept.ctypes.data if kept is not None else None,
                                        low.ctypes.data if low is not None else None)


def _raw_dev(h, with_ptr=True, with_n=True):
    p, n = C.c_void_p(), C.c_uint64()
    return h.lib.cp_batch_ground_device_output(h._h, C.byref(p) if with_ptr else None, C.byref(n) if with_n else None)


@pytest.mark.gpu
def test_state_errors_and_the_run_after():
    cfg = scans.config(2)
    frames = scans.generate(cfg, 4, base_seed=940)
    msgs = _msgs(frames)
    N = sum(len(f) for f in frames)
    with api.ConesGpu(max_points=N, max_frames=4) as h:
        out = np.empty((N, 8), np.float32)
        assert _raw(h, G, out, N) == api.CP_E_STATE                       # nothing staged
        assert _raw_dev(h) == api.CP_E_STATE
        h.set_host_input(msgs)
        runs = []
        for _ in range(2):                                                # direct, then captured into a graph
            h.run(cfg.detect, G)
            runs.append([a.tobytes() for a in h.results()])
        assert runs[0] == runs[1]
        for _ in range(2):
            h.run(cfg.detect, G)
            assert _raw(h, G, out, N) == api.CP_OK
            with pytest.raises(api.ConesGpuError) as e:
                h.results()
            assert e.value.status == api.CP_E_STATE
            with pytest.raises(api.ConesGpuError) as e:
                h.batch_track(api.track_params(False, False))
            assert e.value.status == api.CP_E_STATE
            assert _raw_dev(h) == api.CP_OK
            h.run(cfg.detect, G)                                          # graph replay on the staged input
            assert [a.tobytes() for a in h.results()] == runs[0]
            assert _raw_dev(h) == api.CP_E_STATE                          # a run since the ground call
        assert _raw(h, None, out, N) == api.CP_E_PARAM
        assert _raw(h, G, out, N - 1) == api.CP_E_CAPACITY
        assert _raw(h, G, None, 0) == api.CP_OK                           # device output only: no capacity needed
        assert _raw_dev(h, with_ptr=False) == api.CP_E_PARAM
        assert _raw_dev(h, with_n=False) == api.CP_E_PARAM
        assert _raw_dev(h) == api.CP_OK
        h.set_host_input(msgs)
        assert _raw_dev(h) == api.CP_E_STATE                              # staged since the ground call
        assert _raw(h, G, out, N) == api.CP_OK
        h.ground_remove(msgs[0], G)
        assert _raw_dev(h) == api.CP_E_STATE                              # the single-frame call reuses the buffer
        h.set_host_input(msgs)
        h.run(cfg.detect, G)
        assert [a.tobytes() for a in h.results()] == runs[0]


@pytest.mark.gpu
def test_launch_count_does_not_grow_with_frames():
    cfg = scans.config(2)
    src = scans.generate(cfg, 4, base_seed=950)
    frames = [src[i % 4][(i * 37) % 1000:][:TILE + 1] for i in range(512)]   # every frame crosses a tile
    msgs = _msgs(frames)
    exp = _expect(_views(msgs))
    counts = {}
    with api.ConesGpu(max_points=512 * (TILE + 1), max_frames=512) as h:
        for F in (8, 512):
            h.set_host_input(msgs[:F], fake_missing_intensity=False)
            out, kept, low = h.batch_ground_remove(G)
            _check(out, kept, low, exp[:F])
            counts[F] = h.last_launch_count()
    assert counts[8] == counts[512] > 0, counts


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"CONESGPU_K1_CTAS": "1", "CONESGPU_STREAM_CTAS": "1"}, {"CONESGPU_ROWSKIP": "0"}],
                         ids=["one_cta_per_sm", "no_rowskip"])
def test_launch_geometry(env):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if "CONESGPU_K1_CTAS" in env:
        # 600 frames of two tiles: pass 1 runs one CTA per SM over a contiguous run of tiles, which spans at least
        # two whole frames; pass 2's persistent CTAs take tiles by ticket across frames
        src = scans.generate(scans.config(2), 4, base_seed=960)
        frames = [src[i % 4][(i * 53) % 5000:][:3000] for i in range(600)]
        tiles = sum(-(-len(f) // TILE) for f in frames)
        assert tiles // sms >= 2 * 2, "each pass-1 CTA must cross several frame boundaries"
    else:
        # the default skips rows pass 1 proved to be ground; some rows here are all ground
        frames = list(scans.generate(scans.config(3), 64, base_seed=960))
        keeps = [O.ground_node(O.view_of_xyzi(f), G)[3] for f in frames[:4]]
        assert any((k[:len(k) // 32 * 32].reshape(-1, 32).max(1) == 0).any() for k in keeps)
    msgs = _msgs(frames)
    exp = _expect(_views(msgs))
    F, total = len(frames), sum(len(f) for f in frames)
    with api.ConesGpu(max_points=total, max_frames=F, env=env) as h:
        h.set_host_input(msgs, fake_missing_intensity=False)
        for _ in range(2):
            out, kept, low = h.batch_ground_remove(G)
            _check(out, kept, low, exp)


# ---- the C++ node layer --------------------------------------------------------------------------------------------
def _host_lib():
    from cones_perception_b200.build import HOST_LIB
    lib = C.CDLL(HOST_LIB)
    lib.ch_last_error.restype = C.c_char_p
    lib.ch_ground_create.restype = C.c_void_p
    lib.ch_ground_create.argtypes = [C.c_uint64, C.c_int]
    lib.ch_ground_create_replay.restype = C.c_void_p
    lib.ch_ground_create_replay.argtypes = [C.c_uint64, C.c_uint32, C.c_int]
    lib.ch_ground_destroy.argtypes = [C.c_void_p]
    lib.ch_ground_publish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                      C.c_uint64, C.POINTER(C.c_uint64)]
    return lib


def _publish(lib, gr, frames, replay, intensity):
    xyzi = np.ascontiguousarray(np.concatenate(frames), np.float32)
    n = np.array([len(f) for f in frames], np.uint32)
    out = np.zeros(64 << 20, np.uint8)
    used = C.c_uint64()
    rc = lib.ch_ground_publish(gr, xyzi.ctypes.data, n.ctypes.data, len(frames), intensity, int(replay),
                               out.ctypes.data, out.nbytes, C.byref(used))
    assert rc == 0, lib.ch_last_error()
    return out[:used.value].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("cut", ["max_frames", "max_points"])
@pytest.mark.parametrize("intensity", [1, 0])
def test_cpp_replay_publishes_what_cloud_handler_publishes(cut, intensity):
    lib = _host_lib()
    cfg = scans.config(2)
    src = scans.generate(cfg, 10, base_seed=970)
    frames = [f[:len(f) - 333 * i] for i, f in enumerate(src)]          # ragged
    n = cfg.points_per_frame
    per_msg = lib.ch_ground_create(n, 0)
    # 4 messages per batch (4 + 4 + 2), or at most 2.5 frames of points per batch (2 at a time)
    rep = lib.ch_ground_create_replay(4 * n, 4, 0) if cut == "max_frames" else \
        lib.ch_ground_create_replay(5 * n // 2, 16, 0)
    try:
        assert per_msg and rep, lib.ch_last_error()
        exp = _publish(lib, per_msg, frames, False, intensity)
        got = _publish(lib, rep, frames, True, intensity)
        assert got == exp
        assert _publish(lib, rep, frames[:1], False, intensity) == _publish(lib, per_msg, frames[:1], False, intensity)
        assert _publish(lib, rep, frames[3:], True, intensity) == _publish(lib, per_msg, frames[3:], False, intensity)
    finally:
        lib.ch_ground_destroy(per_msg)
        lib.ch_ground_destroy(rep)
