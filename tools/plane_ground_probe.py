"""The plane ground model against the sector model: `python tools/plane_ground_probe.py OUT_DIR [reps]`.

Config 3, 512 frames, device-resident input, level and pitched batches (every frame pitched and rolled by a seeded
random angle within +-3 deg).  For the sector model and for the plane model at H = 16, 64 and 256 hypotheses: the
step time (host wall clock around cp_batch_run + cp_sync, median of `reps`), the device time of the run (CUDA events),
launches, rows loaded, and whether cp_sync re-ran the back half (the retry grows the launch count).  Also cp_detect's
p50 on one config-3 frame with the plane model.  Next to the times: the bytes-based floor of the plane node (three
passes over 16 B per point plus the 32 B message, then the detector's pass over the 32 B message) at the rate of a
device-to-device copy measured in the same run, and the fp32 work of the scoring pass (3 H FMA per point).  Reports
the card's name and power limit.  Writes one JSON line to OUT_DIR/plane_ground_probe.json."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cones_perception_b200 import api, scans  # noqa: E402
from cones_perception_b200.pointcloud2 import PointCloud2  # noqa: E402

out_dir = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
os.makedirs(out_dir, exist_ok=True)

import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("plane_ground_probe: no CUDA device")

cfg = scans.config(3)
F, N = 512, cfg.points_per_frame
NP = F * N


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def rotate(p, pitch_deg, roll_deg):
    a, b = np.radians(pitch_deg), np.radians(roll_deg)
    Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    Rx = np.array([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]])
    q = p.astype(np.float64)
    q[:, :3] = q[:, :3] @ (Rx @ Ry).T
    return q.astype(np.float32)


def copy_gbps():
    a = torch.empty(NP * 16, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    ts = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return 2 * a.numel() / (np.median(ts) * 1e-3) / 1e9   # read + write


level = scans.generate(cfg, F, base_seed=0)
rng = np.random.default_rng(0)
pitched = np.stack([rotate(f, *rng.uniform(-3, 3, 2)) for f in level])
res = {"card": card(), "frames": F, "points_per_frame": N, "reps": reps, "copy_GBps": copy_gbps(), "runs": []}
gbps = res["copy_GBps"]
# plane node: score + count + write read 16 B/point each, the message is written (32 B/point); then the detector's
# own pass reads the 32 B message
plane_bytes = NP * (3 * 16 + 32 + 32)
res["floor_ms"] = {"sector_two_passes_16B": 2 * NP * 16 / gbps / 1e6, "plane_chain": plane_bytes / gbps / 1e6}

for name, frames in (("level", level), ("pitched", pitched)):
    dev = torch.from_numpy(np.ascontiguousarray(frames.reshape(-1, 4))).cuda()
    for H in (None, 16, 64, 256):
        # a fresh handle per model: a back-half retry leaves the handle on the bigger variant for later runs
        with api.ConesGpu(max_points=NP, max_frames=F) as h:
            h.set_device_input(dev.data_ptr(), [N] * F, 16, (0, 4, 8, 12), keep=dev)
            h.set_ground_plane(None if H is None else api.plane_params(seed=0, n_hypotheses=H))
            h.run(cfg.detect, cfg.ground)
            before = h.last_launch_count()
            h.sync()
            retried = h.last_launch_count() != before
            for _ in range(3):
                h.run(cfg.detect, cfg.ground)
                h.sync()
            wall, dev_ms = [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                h.run(cfg.detect, cfg.ground)
                h.sync()
                wall.append((time.perf_counter() - t0) * 1e3)
                dev_ms.append(h.last_run_ms())
            ctr, _, cl = h.results()
            run = {"batch": name, "model": "sector" if H is None else "plane", "H": H,
                   "step_ms_p50": float(np.median(wall)), "device_ms_p50": float(np.median(dev_ms)),
                   "launches": h.last_launch_count(), "rows_loaded": h.last_rows_loaded(),
                   "back_half_retry": bool(retried), "clusters": int(len(cl)),
                   "mean_ground_kept": float(ctr["n_ground_kept"].mean()),
                   "mean_cropped": float(ctr["n_cropped"].mean())}
            if H is not None:
                run["scoring_fma_per_point"] = 3 * H
                run["scoring_tflop"] = 2 * 3 * H * NP / 1e12
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
    del dev

one = PointCloud2.from_xyzi(np.ascontiguousarray(pitched[0]))
with api.ConesGpu(max_points=N, max_frames=1) as h:
    h.set_ground_plane(api.plane_params(seed=0, n_hypotheses=64))
    for _ in range(5):
        h.detect(one, cfg.detect, cfg.ground)
    ts = []
    for _ in range(max(reps, 50)):
        t0 = time.perf_counter()
        h.detect(one, cfg.detect, cfg.ground)
        ts.append((time.perf_counter() - t0) * 1e3)
    res["cp_detect_plane_H64_p50_ms"] = float(np.median(ts))
    res["cp_detect_plane_H64_launches"] = h.last_launch_count()

with open(os.path.join(out_dir, "plane_ground_probe.json"), "w") as f:
    f.write(json.dumps(res) + "\n")
print(json.dumps({k: v for k, v in res.items() if k != "runs"}))
