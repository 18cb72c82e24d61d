"""Colours of a fused run from the ground node's messages: `python tools/groundless_colors_probe.py OUT_DIR [reps]`.

Config 3, 512 frames, device-resident input, colour net loaded.  Three ways to get every cluster's colour:
  (a) fused run (ground removal inside) + cp_batch_cone_colors with CP_COLOR_CLOUD_STAGED: crops from the raw scan
  (b) the same run + cp_batch_cone_colors with CP_COLOR_CLOUD_GROUNDLESS: crops from the ground node's messages
  (c) the two-handle device chain of the reference's launch: cp_batch_ground_remove (device output), a second handle
      on the 32-byte messages, a run without ground removal, then cp_batch_cone_colors
(b) and (c) must give identical colours, flags, counts and probabilities.  Reports how many crops differ between (a)
and (b).  Times are medians of `reps` host wall-clock measurements of calls that end in a device synchronise: the
colour call alone for (a) and (b); for (c) the ground call, the chained run and its colour call, together and apart.
Reports the card's name and power limit.  Writes one JSON line to OUT_DIR/groundless_colors_probe.json."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cones_perception_b200 import api, scans  # noqa: E402

out_dir = sys.argv[1]
reps = max(10, int(sys.argv[2]) if len(sys.argv) > 2 else 10)
os.makedirs(out_dir, exist_ok=True)

import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("groundless_colors_probe: no CUDA device")

cfg = scans.config(3)
F, N = 512, cfg.points_per_frame
g = cfg.ground
frames = scans.generate(cfg, F, base_seed=0)
frames[..., 3] = np.clip(frames[..., 3] * 2.5, 0, 255)   # the intensity range the classifier was trained on
dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()
NP = F * N
model = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                             "dam_net_model.npz"))["tflite"].tobytes()


def med(v):
    return float(np.median(v))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def timed(fn):
    t = time.perf_counter()
    out = fn()       # every call timed here ends in a device synchronise
    return (time.perf_counter() - t) * 1e3, out


result = {"config": 3, "frames": F, "points": NP, "reps": reps}
with api.ConesGpu(max_points=NP, max_frames=F) as h, api.ConesGpu(max_points=NP, max_frames=F) as a, \
        api.ConesGpu(max_points=NP, max_frames=F, max_point_step=32) as b:
    h.color_net_load_tflite(model)
    b.color_net_load_tflite(model)
    h.set_device_input(dev.data_ptr(), np.full(F, N, np.uint32), keep=dev)
    h.run(cfg.detect, g)
    _, off, cl = h.results()
    t_a, t_b = [], []
    for r in range(reps + 1):      # (a) and (b) alternate; repetition 0 warms up (buffers grow)
        h.set_color_cloud(False)
        ta, col_a = timed(h.batch_cone_colors)
        h.set_color_cloud(True)
        tb, col_b = timed(h.batch_cone_colors)
        if r:
            t_a.append(ta)
            t_b.append(tb)
    launches = h.last_launch_count()

    a.set_device_input(dev.data_ptr(), np.full(F, N, np.uint32), keep=dev)

    t_g, t_r, t_c, t_all = [], [], [], []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        tg, _ = timed(lambda: a.batch_ground_remove(g, host=False))
        ptr, n = a.ground_device_output()
        assert n == NP

        def run_b():
            b.set_device_input(ptr, np.full(F, N, np.uint32), 32, (0, 4, 8, 16))
            b.run(cfg.detect, None)
            b.sync()
        tr, _ = timed(run_b)
        tc, col_c = timed(b.batch_cone_colors)
        tall = (time.perf_counter() - t0) * 1e3
        if r:
            t_g.append(tg)
            t_r.append(tr)
            t_c.append(tc)
            t_all.append(tall)
    _, coff, ccl = b.results()

assert np.array_equal(off, coff) and np.array_equal(cl.view(np.uint32), ccl.view(np.uint32)), "records differ"
assert np.array_equal(col_b[0], col_c[0]), "colours differ"
assert np.array_equal(col_b[1].view(np.uint32), col_c[1].view(np.uint32)), "probabilities differ"
assert np.array_equal(col_b[2], col_c[2]), "flags differ"
assert np.array_equal(col_b[3], col_c[3]), "counts differ"
result.update({
    "clusters": int(len(cl)), "b_equals_c": True,
    "crops_differing_a_b": int((col_a[3] != col_b[3]).sum()),
    "colours_differing_a_b": int((col_a[0] != col_b[0]).sum()),
    "crop_points_a": int(col_a[3].sum()), "crop_points_b": int(col_b[3].sum()),
    "a_staged_colors_ms": med(t_a), "b_groundless_colors_ms": med(t_b), "colour_call_launches": launches,
    "c_chain_total_ms": med(t_all), "c_ground_ms": med(t_g), "c_run_ms": med(t_r), "c_colors_ms": med(t_c),
})
result["gpu"], result["power_limit"] = card()
print(json.dumps(result))
with open(os.path.join(out_dir, "groundless_colors_probe.json"), "w") as f:
    f.write(json.dumps(result) + "\n")
