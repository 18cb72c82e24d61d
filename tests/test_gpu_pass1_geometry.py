"""-m gpu: pass 1 and the per-frame kernel give the same results at every grid cap.

Pass 1 (`ground_sector_min_kernel`) refreshes its prefilter bounds per warp without a barrier and drops whole rows
whose lowest key is not below the all-sector bound, so its sector minima must not depend on how tiles are spread
over CTAs (`CONESGPU_K1_CTAS`), and the per-frame kernel's results not on how many frames each CTA takes
(`CONESGPU_FRAME_CTAS`).  Every case compares counters, cluster offsets, cluster records and (through the tap) the
per-sector minima with the CPU oracle bit for bit, on a config-3 batch and on scenes built against the row
prefilter: rows of one z, axis points and signed zeros, NaN and inf inside rows, a frame whose lowest point is its
last, ragged frame sizes.
"""
import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200.pointcloud2 import PointCloud2
from oracle import oracle as O
from tests.util import boundary_cloud

pytestmark = pytest.mark.gpu

_COUNTERS = ("n_ground_kept", "n_cropped", "n_voxels", "n_components", "key_bits")
_CFG = scans.config(3)
_BATCHES, _ORACLE = {}, {}


def _batch(name):
    if name in _BATCHES:
        return _BATCHES[name]
    cfg = _CFG
    if name == "cfg3":
        frames = list(scans.generate(cfg, 6, base_seed=4400))
    else:
        base = scans.generate(cfg, 4, base_seed=4401)
        rng = np.random.default_rng(4402)
        frames = []
        # a flat sheet: whole 32-point rows of one z, so every row's lowest key equals a sector minimum
        flat = np.array(base[0][:5 * 2048])
        flat[:, 2] = np.float32(-0.6)
        flat[rng.choice(len(flat), 300, replace=False), 2] = np.float32(0.4)
        frames.append(flat)
        # axis points, signed zeros, sector boundaries, NaN and inf (tests/util.py)
        frames.append(boundary_cloud(cfg.detect, seed=4403, n_random=6000))
        # NaN and inf inside otherwise ordinary rows, and a row that holds the frame's lowest point next to a NaN
        f = np.array(base[1][:7 * 2048 + 5])
        f[[5, 40, 77, 2049], 2] = [np.nan, np.inf, -np.inf, -np.nan]
        f[[100, 101], 0] = [np.nan, np.inf]
        f[[130, 131], 1] = [-np.inf, np.nan]
        f[133, 2] = f[:, 2][np.isfinite(f[:, 2])].min() - np.float32(0.3)
        frames.append(f)
        # the lowest point of the frame is its last one (alone in the last, partial row)
        g = np.array(base[2][:3 * 2048 + 33])
        g[-1, :3] = [-2.5, -1.0, g[:, 2].min() - np.float32(0.5)]
        frames.append(g)
        # ragged sizes around rows and tiles
        for n in (1, 31, 33, 2047, 2049):
            frames.append(np.array(base[3][rng.integers(0, 1000):][:n]))
    _BATCHES[name] = [np.ascontiguousarray(f, np.float32) for f in frames]
    return _BATCHES[name]


def _expected(name):
    if name not in _ORACLE:
        cls, ctrs, lows = [], [], []
        for f in _batch(name):
            cl, octr, _ = O.detect(O.view_of_xyzi(f), _CFG.detect, _CFG.ground, O.CANONICAL)
            cls.append(cl)
            ctrs.append([octr.n_ground_kept, octr.n_cropped, octr.n_voxels, octr.n_components, octr.key_bits])
            lows.append(np.asarray(O.ground_minima(O.points32(f), _CFG.ground.default_lowest_point), np.float32))
        off = np.concatenate([[0], np.cumsum([len(c) for c in cls])]).astype(np.uint32)
        _ORACLE[name] = (off, np.concatenate(cls), np.array(ctrs, np.int64), np.stack(lows))
    return _ORACLE[name]


def _check(res, name, tag):
    ctr, off, cl = res
    e_off, e_cl, e_ctr, _ = _expected(name)
    got = np.stack([ctr[n].astype(np.int64) for n in _COUNTERS], 1)
    for j, n in enumerate(_COUNTERS):
        bad = np.nonzero(got[:, j] != e_ctr[:, j])[0]
        assert len(bad) == 0, (tag, n, "frames", bad[:8], got[bad[:8], j], e_ctr[bad[:8], j])
    assert np.array_equal(off, e_off), (tag, "cluster offsets")
    assert np.array_equal(cl.view(np.uint32), e_cl.view(np.uint32)), (tag, "clusters not bit-exact")


def _capacity(name):
    frames = _batch(name)
    return sum(len(f) for f in frames), len(frames)


def _run(h, name):
    h.set_host_input([PointCloud2.from_xyzi(f) for f in _batch(name)])
    h.run(_CFG.detect, _CFG.ground)
    return h.results()


CAPS = {f"k1_{k}": {"CONESGPU_K1_CTAS": str(k)} for k in (1, 2, 4, 8)}
CAPS.update({f"frame_{k}": {"CONESGPU_FRAME_CTAS": str(k)} for k in (1, 2, 4)})


@pytest.mark.parametrize("batch", ["cfg3", "stress"])
@pytest.mark.parametrize("cap", list(CAPS))
def test_grid_caps_match_oracle_with_sector_minima(batch, cap):
    n, F = _capacity(batch)
    with api.ConesGpu(max_points=n, max_frames=F, taps=True, env=CAPS[cap]) as h:
        res = _run(h, batch)
        low = h.tap(api.TAP_SECTOR_LOW).reshape(-1, 17)
    _check(res, batch, cap)
    assert np.array_equal(low.view(np.uint32), _expected(batch)[3].view(np.uint32)), (cap, "sector minima")
