"""The sector model's ground counts when a batch is retried into the general back half.

With ground removal the per-frame kernel evaluates pass 2 itself and stores each frame's ground survivors G_f.  A frame
that then overflows the per-frame kernel is re-run through the general back half, whose pass over the scan counts the
ground survivors again; the counts are cleared first, so n_ground_kept stays G_f, and so does the multiplicity of the
padding points the ground node appends (part of a voxel mean when the padding survives the crop)."""
import dataclasses

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200.params import GroundParams
from cones_perception_b200.pointcloud2 import PointCloud2
from oracle import oracle as O

G = GroundParams()
CTR = ("n_points", "n_ground_kept", "n_cropped", "n_voxels", "n_components", "n_clusters")


def _pitched(n, seed, cfg):
    """Frames pitched and rolled by up to 3 deg: the far ground rises above the sector minima, and tens of thousands
    of points per frame survive, more than the per-frame back half holds."""
    rng = np.random.default_rng(seed)
    out = []
    for f in scans.generate(cfg, n, base_seed=seed):
        a, b = np.radians(rng.uniform(-3, 3, 2))
        Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        Rx = np.array([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]])
        q = f.astype(np.float64)
        q[:, :3] = q[:, :3] @ (Rx @ Ry).T
        out.append(np.ascontiguousarray(q.astype(np.float32)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("pad_survives", [False, True])
def test_retry_into_the_general_path_keeps_the_ground_counts(pad_survives):
    cfg = scans.config(3)
    d = dataclasses.replace(cfg.detect, distance_treshold_min=0.0) if pad_survives else cfg.detect
    frames = _pitched(3, 91, cfg)
    msgs = [PointCloud2.from_xyzi(f) for f in frames]
    with api.ConesGpu(max_points=sum(len(f) for f in frames), max_frames=len(frames)) as h:
        h.set_host_input(msgs)
        h.run(d, G)
        before = h.last_launch_count()
        h.sync()
        assert h.last_launch_count() > before, "the batch did not take the back-half retry"
        ctr, off, cl = h.results()
    for f, m in enumerate(msgs):
        e, octr, _ = O.detect(O.view_of_msg(m, True), d, G, O.CANONICAL)
        assert np.array_equal(cl[off[f]:off[f + 1]].view(np.uint32), e.view(np.uint32)), f
        exp = {k: getattr(octr, k) for k in CTR}
        if pad_survives and octr.n_points > octr.n_ground_kept:
            # the N - G filler points that survive the crop are one record with a multiplicity on the GPU (as in
            # tests/util.py assert_frame_parity); the oracle materialises them
            exp["n_cropped"] -= octr.n_points - octr.n_ground_kept - 1
        for k in CTR:
            assert int(ctr[k][f]) == exp[k], (f, k, int(ctr[k][f]), exp[k])
