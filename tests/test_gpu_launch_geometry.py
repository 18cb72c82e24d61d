"""-m gpu: results must not depend on launch geometry.

The host sizes most grids from a guess, not from the work: the general back half from the previous run's survivor
and voxel counts (`hinted`, pipeline.cu), a run replayed from a CUDA graph with the grids of the run it was captured
on, the sort passes at one CTA per tile up to a cap (radix_sort.cuh), and six switches change grids or swap whole
kernels.  That is correct only because every kernel loops over device-resident bounds and draws its work by ticket.
These cases put that claim where it is thin: many tickets per CTA, grids far larger than the work, a graph frozen
on sparse grids and replayed on dense data, sorts past the grid cap, frames and pass-1 chunks shared between CTAs.
Every case compares with the CPU oracle bit for bit and asserts, from sizes it can see, that it really reaches the
grid-to-work ratio it is named after.
"""
import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200.params import GroundParams
from cones_perception_b200.pointcloud2 import PointCloud2
from oracle import oracle as O
from tests.util import assert_frame_parity, oracle_stages, run_batch_with_taps

pytestmark = pytest.mark.gpu

TILE = 2048            # kSortTile (radix_sort.cuh) = kStreamTile (stream_kernels.cuh) = 2048 items


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tiles(n):
    return (int(n) + TILE - 1) // TILE


def _hinted_work(hint):
    """pipeline.cu `hinted()`: after a run with `hint` > 0 survivors the general back half sizes its grids for
    2 * hint + 8192 items; the voxel sort then gets one CTA per 2048 of them (radix_sort.cuh radix_sort_passes)."""
    return 2 * int(hint) + 8192


# ---- the oracle, cached per input (the switch matrix reuses the same batches) ----------------------------------

_ORACLE = {}


def _expected(name, frames, d, g):
    """(cluster offsets, all clusters, per-frame counters) of the oracle for a batch, computed once per name."""
    if name not in _ORACLE:
        cls, ctrs = [], []
        for f in frames:
            cl, octr, _ = O.detect(O.view_of_xyzi(np.ascontiguousarray(f)), d, g, O.CANONICAL)
            cls.append(cl)
            ctrs.append([octr.n_ground_kept, octr.n_cropped, octr.n_voxels, octr.n_components, octr.key_bits])
        off = np.concatenate([[0], np.cumsum([len(c) for c in cls])]).astype(np.uint32)
        _ORACLE[name] = (off, np.concatenate(cls), np.array(ctrs, np.int64))
    return _ORACLE[name]


_COUNTERS = ("n_ground_kept", "n_cropped", "n_voxels", "n_components", "key_bits")


def _assert_matches_oracle(res, exp, tag):
    ctr, off, cl = res
    e_off, e_cl, e_ctr = exp
    got = np.stack([ctr[n].astype(np.int64) for n in _COUNTERS], 1)
    for j, n in enumerate(_COUNTERS):
        bad = np.nonzero(got[:, j] != e_ctr[:, j])[0]
        assert len(bad) == 0, (tag, n, "frames", bad[:8], got[bad[:8], j], e_ctr[bad[:8], j])
    assert np.array_equal(off, e_off), (tag, "cluster offsets")
    assert np.array_equal(cl.view(np.uint32), e_cl.view(np.uint32)), (tag, "clusters not bit-exact")


def _same_bytes(a, b):
    return all(x.tobytes() == y.tobytes() for x, y in zip(a, b))


def _push_out(frame, centre, half_width):
    """The frame with every point outside the wedge |angle - centre| < half_width pushed 20 m further out along
    its own bearing (same sector, same height, so the ground minima barely move): beyond every preset's
    distance_treshold_max, so only the wedge can survive the crop."""
    x, y = frame[:, 0].astype(np.float64), frame[:, 1].astype(np.float64)
    ang = np.angle(np.exp(1j * (np.arctan2(y, x) - centre)))
    r = np.hypot(x, y)
    s = np.where(np.abs(ang) < half_width, 1.0, 1.0 + 20.0 / np.maximum(r, 0.01))
    out = frame.copy()
    out[:, 0] = (x * s).astype(np.float32)
    out[:, 1] = (y * s).astype(np.float32)
    return out


def _dense_and_sparse_cfg4():
    """One config-4 frame (2.62 M points, 261 k crop survivors) and the same frame with a few hundred survivors."""
    cfg = scans.config(4)
    dense = scans.generate(cfg, 1, base_seed=0)[0]
    return cfg, dense, _push_out(dense, 0.3025, 0.0025)


def _cfg3_sparse(frames, cfg):
    """Config-3 frames cut down to the points around their first cone: a handful of crop survivors each."""
    out = []
    for f in frames:
        cl, _, _ = O.detect(O.view_of_xyzi(f), cfg.detect, cfg.ground, O.CANONICAL)
        out.append(_push_out(f, float(np.arctan2(cl["y"][0], cl["x"][0])), 0.01))
    return np.stack(out)


# ---- 1. sorts past the grid cap -----------------------------------------------------------------------------------

def _sort_keys(n, bits, seed):
    rng = np.random.default_rng(seed)
    keys = rng.integers(0, 1 << min(bits, 63), n, dtype=np.uint64)
    if bits == 64:
        keys |= rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63)
    keys[::3] = keys[0]                     # one key a third of the time, in every tile: stability across tiles
    keys[1::7] = keys[1]
    # bits 8..15 are the same for every key: the second pass sees a single digit
    keys = (keys & ~np.uint64(0xFF00)) | np.uint64(0x5A00)
    m = min(n // 4, 3 * TILE + 17)
    run = np.sort(keys[:m])
    keys[n // 4:n // 4 + m] = run           # an already sorted run, several tiles long
    keys[n // 2:n // 2 + m] = run[::-1]     # and the same run reversed
    return keys


# radix_sort.cuh radix_sort_enqueue (cp_debug_sort): grid = min(tiles, SMs * 16), or SMs * 3 with persistent CTAs
# (CONESGPU_TILE_CTAS=0); every CTA draws tiles by ticket until they run out.
_SORT_GRIDS = {"per_tile": ({}, 16), "persistent": ({"CONESGPU_TILE_CTAS": "0"}, 3)}


def _sort_sizes(sms, per_sm):
    cap = per_sm * sms * TILE
    looping = 5 * cap // 2 + 1001 if per_sm == 16 else 3_000_017   # 12.1 M / 3.0 M items on 148 SMs
    return {"grid_equals_tiles": cap, "one_second_ticket": cap + 1, "every_cta_loops": looping}


@pytest.fixture(scope="module", params=list(_SORT_GRIDS))
def sorter(request, sms):
    env, per_sm = _SORT_GRIDS[request.param]
    n_max = max(_sort_sizes(sms, per_sm).values())
    # cp_debug_sort needs n <= max_voxels (= max_points + max_frames here)
    with api.ConesGpu(max_points=n_max, max_frames=1, env=env) as h:
        yield h, per_sm


@pytest.mark.parametrize("bits", [24, 64])
@pytest.mark.parametrize("size", ["grid_equals_tiles", "one_second_ticket", "every_cta_loops"])
def test_sort_past_the_grid_cap_matches_stable_argsort(sorter, sms, size, bits):
    h, per_sm = sorter
    n = _sort_sizes(sms, per_sm)[size]
    grid = min(_tiles(n), per_sm * sms)
    if size == "grid_equals_tiles":
        assert _tiles(n) == grid
    elif size == "one_second_ticket":
        assert _tiles(n) == grid + 1
    else:
        assert _tiles(n) > 2 * grid, (n, grid)
    keys = _sort_keys(n, bits, seed=n + bits)
    assert len(np.unique((keys >> np.uint64(8)) & np.uint64(0xFF))) == 1       # the single-digit pass
    vals = np.arange(n, dtype=np.uint32)
    k, v = h.debug_sort(keys, vals, bits)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(k, keys[order])
    assert np.array_equal(v, order.astype(np.uint32))


# ---- 2. the size hint carried between direct runs, checked stage by stage -----------------------------------------

_STAGES = {}


def _stages(name, frame, d, g):
    if name not in _STAGES:
        _STAGES[name] = (oracle_stages(frame, d, g), O.detect(O.view_of_xyzi(frame), d, g, O.CANONICAL)[1].key_bits)
    return _STAGES[name]


def test_size_hint_from_sparse_runs_and_dense_runs_stage_by_stage():
    """One general-back-half handle with taps on (no graphs: every run is direct), so each run's grids come from the
    run before it: sparse -> dense -> sparse -> dense -> 8 config-3 frames -> sparse.  A dense frame after a sparse one
    sorts ~128 tiles with 5 CTAs; a sparse run after a dense one has hundreds of idle CTAs drawing tickets past the end."""
    cfg4, dense, sparse = _dense_and_sparse_cfg4()
    cfg3 = scans.config(3)
    eight = list(scans.generate(cfg3, 8, base_seed=3100))
    runs = [("sparse", [sparse], cfg4.detect, None), ("dense", [dense], cfg4.detect, None),
            ("sparse", [sparse], cfg4.detect, None), ("dense", [dense], cfg4.detect, None),
            ("eight", eight, cfg3.detect, cfg3.ground), ("sparse", [sparse], cfg4.detect, None)]
    with api.ConesGpu(max_points=len(dense), max_frames=8, taps=True, back_mode=3) as h:
        prev = None                                         # survivors of the previous run: the hint
        for rep, (name, frames, d, g) in enumerate(runs):
            ctr, k_off, clusters, offs, taps = run_batch_with_taps(h, frames, d, g)
            for f, a in enumerate(frames):
                ora, key_bits = _stages(f"{name}/{f}", a, d, g)
                assert_frame_parity(h, f, ora, offs, taps, ctr, k_off, clusters)
                assert int(ctr["key_bits"][f]) == key_bits, (rep, name, f)
            n = int(ctr["n_cropped"].sum())
            assert n > 0, "the hint only moves after a run with survivors"
            if prev is not None:
                work = _hinted_work(prev)
                if name == "dense":        # the grids of a sparse run: every sort CTA takes 16 tickets or more
                    assert n >= 16 * work, (rep, n, prev)
                else:                      # the grids of a bigger run: at least 4 times more sort CTAs than tiles
                    assert _tiles(work) >= 4 * _tiles(n), (rep, n, prev)
            prev = n


# ---- 3. a graph frozen on sparse grids, replayed on dense data ----------------------------------------------------

def _replay_sequence(h, dev, inputs, d, g, exp):
    """Writes each input into the device buffer in place, runs, and checks the run against the oracle."""
    import torch
    out, launches = [], []
    for rep, name in enumerate(["sparse", "sparse", "sparse", "dense", "dense", "sparse", "dense"]):
        dev.copy_(torch.from_numpy(inputs[name]))
        torch.cuda.synchronize()
        h.run(d, g)
        res = h.results()
        _assert_matches_oracle(res, exp[name], (rep, name))
        out.append((name, res))
        launches.append(h.last_launch_count())
    # direct run, capture, then replays only: the key never changes, so the graph is never captured again
    assert len(set(launches[1:])) == 1, launches
    for name in ("sparse", "dense"):
        same = [r for n, r in out if n == name]
        assert all(_same_bytes(same[0], r) for r in same[1:]), name
    return out


def test_graph_captured_on_a_sparse_frame_replays_dense_frames():
    import torch
    cfg, dense, sparse = _dense_and_sparse_cfg4()
    inputs = {"dense": dense, "sparse": sparse}
    exp = {k: _expected(f"cfg4/{k}", [v], cfg.detect, None) for k, v in inputs.items()}
    n_sparse, n_dense = int(exp["sparse"][2][0, 1]), int(exp["dense"][2][0, 1])
    # the graph is captured on the second run, whose grids come from the first (sparse) run's survivors
    assert 0 < n_sparse and n_dense >= 16 * _hinted_work(n_sparse), (n_sparse, n_dense)
    dev = torch.from_numpy(np.ascontiguousarray(sparse)).cuda()
    with api.ConesGpu(max_points=len(dense), max_frames=1, back_mode=3) as h:
        h.set_device_input(dev.data_ptr(), np.array([len(dense)], np.uint32), keep=dev)
        _replay_sequence(h, dev, inputs, cfg.detect, None, exp)


def test_graph_captured_on_a_sparse_batch_replays_dense_batches():
    """A uniform batch of config-3 frames with ground removal.  (64 frames: the survivors of 4 dense frames would fit
    the 8192 items the hint adds anyway, and the sort grid would never be short.)"""
    import torch
    cfg = scans.config(3)
    F = 64
    dense = scans.generate(cfg, F, base_seed=3200)
    sparse = _cfg3_sparse(dense, cfg)
    inputs = {"dense": dense, "sparse": sparse}
    exp = {k: _expected(f"cfg3x{F}/{k}", v, cfg.detect, cfg.ground) for k, v in inputs.items()}
    n_sparse, n_dense = int(exp["sparse"][2][:, 1].sum()), int(exp["dense"][2][:, 1].sum())
    assert n_sparse > 0 and (exp["sparse"][2][:, 1] < 200).all()
    # the frozen voxel sort has ceil(work / 2048) CTAs; the dense batch gives each of them at least two tiles
    assert _tiles(n_dense) >= 2 * _tiles(_hinted_work(n_sparse)), (n_sparse, n_dense)
    dev = torch.from_numpy(np.ascontiguousarray(sparse)).cuda()
    with api.ConesGpu(max_points=F * cfg.points_per_frame, max_frames=F, back_mode=3) as h:
        h.set_device_input(dev.data_ptr(), np.full(F, cfg.points_per_frame, np.uint32), keep=dev)
        _replay_sequence(h, dev, inputs, cfg.detect, cfg.ground, exp)


# ---- 4. every grid-cap switch against the default -----------------------------------------------------------------

SWITCHES = {
    "baseline": {},
    "tile_ctas_0": {"CONESGPU_TILE_CTAS": "0"},
    "stream_ctas_1": {"CONESGPU_STREAM_CTAS": "1"},
    "k1_ctas_1": {"CONESGPU_K1_CTAS": "1"},
    "frame_ctas_1": {"CONESGPU_FRAME_CTAS": "1"},
    "fused_front": {"CONESGPU_FUSED_FRONT": "1"},
    "prio": {"CONESGPU_PRIO": "1"},
    "all_caps": {"CONESGPU_STREAM_CTAS": "1", "CONESGPU_K1_CTAS": "1", "CONESGPU_FRAME_CTAS": "1",
                 "CONESGPU_TILE_CTAS": "0"},
}

N_SMALL = 5 * TILE     # points per frame of the small-frame batches: 5 stream tiles
F_SMALL = 600          # frames: more than 148 SMs x 4 per-frame-kernel CTAs


_BATCHES = {}


def _small_batch(name):
    """600 config-3 scans cut to 5-beam rings (10 240 points, 5 stream tiles each): 10 scans x 60 ring offsets.
    "ragged" cuts the same rings to random lengths, with empty frames (first and last too), one-point, one-tile,
    exactly-2048 and 2049-point frames."""
    if name not in _BATCHES:
        cfg = scans.config(3)
        base = scans.generate(cfg, 10, base_seed=3300)
        frames = [np.ascontiguousarray(base[f % 10][(f // 10) * cfg.az:][:N_SMALL]) for f in range(F_SMALL)]
        if name == "ragged":
            rng = np.random.default_rng(3301)
            n = rng.integers(0, N_SMALL + 1, F_SMALL)
            n[[0, 7, 300, F_SMALL - 1]] = 0
            n[[1, 50]] = 1
            n[[2, 51]] = TILE - 1
            n[[3, 52, 400]] = TILE
            n[[4, 53]] = TILE + 1
            frames = [f[:k] for f, k in zip(frames, n)]
        _BATCHES[name] = (frames, [PointCloud2.from_xyzi(f) for f in frames])
    return _BATCHES[name]


def _pass1_min_boundaries(sizes, grid):
    """Pass 1 (stream_kernels.cuh ground_sector_min_kernel) gives CTA b the contiguous tiles [b*per, (b+1)*per),
    per = ceil(tiles / grid); an empty frame owns one tile (pipeline.cu set_geometry).  Returns the fewest frame
    boundaries any CTA's chunk crosses."""
    tiles_of = np.maximum(1, (np.asarray(sizes) + TILE - 1) // TILE)
    tile_frame = np.repeat(np.arange(len(sizes)), tiles_of)
    per = -(-len(tile_frame) // grid)
    chunks = [tile_frame[b:b + per] for b in range(0, len(tile_frame), per)]
    return min(int(c[-1] - c[0]) for c in chunks[:-1])


_BASELINE = {}


def _run3(switch, mode, batch, g):
    """Direct run, graph capture, replay on one handle: the three must agree byte for byte."""
    frames, msgs = _small_batch("ragged" if batch == "ragged" else "uniform")
    d = scans.config(3).detect
    with api.ConesGpu(max_points=F_SMALL * N_SMALL, max_frames=F_SMALL, back_mode=mode, env=SWITCHES[switch]) as h:
        runs = []
        for _ in range(3):
            ctr, off, cl = h.detect_batch(msgs, d, g)
            runs.append((ctr.copy(), off.copy(), cl.copy()))
    for r in runs[1:]:
        assert _same_bytes(runs[0], r), (switch, mode, batch, "direct run, capture and replay differ")
    return runs[0], frames


@pytest.mark.parametrize("batch", ["uniform", "ragged", "no_ground"])
@pytest.mark.parametrize("mode", [None, 3], ids=["default_back", "general_back"])
@pytest.mark.parametrize("switch", list(SWITCHES))
def test_grid_cap_switch_matches_default_and_oracle(sms, switch, mode, batch):
    cfg = scans.config(3)
    g = None if batch == "no_ground" else cfg.ground
    env = SWITCHES[switch]
    frames, _ = _small_batch("ragged" if batch == "ragged" else "uniform")
    sizes = [len(f) for f in frames]
    # preconditions, from the shapes alone
    assert F_SMALL > 4 * sms        # default per-frame kernel: at most 4 CTAs per SM (DESIGN.md §4.1): CTAs reuse
    if env.get("CONESGPU_FRAME_CTAS") == "1" and mode is None:
        assert F_SMALL >= 4 * sms   # grid = min(frames, SMs x 1): every CTA runs 4 frames or more
    if (env.get("CONESGPU_STREAM_CTAS") == "1" or env.get("CONESGPU_K1_CTAS") == "1") and g is not None:
        # pass-1 grid = min(tiles, SMs x 1) (pipeline.cu grid_for / launch_sector_min)
        assert _pass1_min_boundaries(sizes, sms) >= 2, "each pass-1 CTA must cross two frame boundaries"
    if switch == "fused_front":
        # pipeline.cu enqueue_pipeline: front_fused_kernel runs for a uniform batch with ground removal only
        fused = len(set(sizes)) == 1 and sizes[0] > 0 and g is not None
        assert fused == (batch == "uniform")
    res, _ = _run3(switch, mode, batch, g)
    _assert_matches_oracle(res, _expected(f"small/{batch}", frames, cfg.detect, g), (switch, mode, batch))
    if env.get("CONESGPU_TILE_CTAS") == "0" and mode == 3 and batch == "no_ground":
        # persistent sort passes: 3 CTAs per SM, each loops over several tiles of the voxel sort
        assert _tiles(res[0]["n_cropped"].sum()) > 2 * 3 * sms, int(res[0]["n_cropped"].sum())
    key = (mode, batch)
    if key not in _BASELINE:
        _BASELINE[key] = res if switch == "baseline" else _run3("baseline", mode, batch, g)[0]
    assert _same_bytes(res, _BASELINE[key]), (switch, mode, batch, "differs from the default grids")


def test_ground_node_with_one_pass1_cta_per_sm(sms):
    """cp_ground_remove's pass 1 under CONESGPU_K1_CTAS=1 (with CONESGPU_STREAM_CTAS=1): SMs CTAs, each over a
    contiguous run of tiles, on a cloud of eight config-2 scans.  (cp_ground_remove sizes pass 1 at 8 CTAs per SM
    whatever CONESGPU_STREAM_CTAS says, pipeline.cu; CONESGPU_K1_CTAS overrides that grid in launch_sector_min.)"""
    cfg = scans.config(2)
    cloud = np.ascontiguousarray(scans.generate(cfg, 8, base_seed=3400).reshape(-1, 4))
    assert _tiles(len(cloud)) >= 2 * sms, "every pass-1 CTA must take several tiles"
    msg = PointCloud2.from_xyzi(cloud)
    exp, ekept, elow, _ = O.ground_node(O.view_of_xyzi(cloud), GroundParams())
    e = np.stack([exp[n] for n in ("x", "y", "z", "pad", "intensity", "c1", "c2", "c3")], 1)
    with api.ConesGpu(max_points=len(cloud), env={"CONESGPU_STREAM_CTAS": "1", "CONESGPU_K1_CTAS": "1"}) as h:
        for _ in range(2):
            out, kept, low = h.ground_remove(msg, GroundParams())
            assert kept == ekept
            assert np.array_equal(low.view(np.uint32), elow.view(np.uint32))
            assert np.array_equal(out.view(np.uint32), e.view(np.uint32))
