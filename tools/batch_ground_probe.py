"""The ground node's messages for a whole batch: `python tools/batch_ground_probe.py OUT_DIR [reps]`.

Config 3, 512 frames.  Compares three ways to get every frame's groundless_cloud message:
  (a) cp_batch_ground_remove, device output only, on device-resident input
  (b) cp_batch_ground_remove with host output (survivors copied back, padding written by the host), on the same input
  (c) the per-frame loop it replaces: cp_ground_remove on each frame's pageable message, one handle
The outputs of (a) and (b) must equal (c) byte for byte.  Times are host wall clock around calls that end in a device
synchronise (medians of `reps`), plus the device time of (a) with CUDA events on the handle's stream.  Next to them:
the bytes the call must move (pass 1 reads 16 B per point, pass 2 reads 16 B per point of the rows it could not skip,
the messages write 32 B per point) over the rate of a device-to-device copy measured in the same run, which is the
floor.  Reports the card's name and power limit.  Writes one JSON line to OUT_DIR/batch_ground_probe.json."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cones_perception_b200 import api, scans  # noqa: E402
from cones_perception_b200.params import to_c_ground  # noqa: E402
from cones_perception_b200.pointcloud2 import PointCloud2  # noqa: E402

out_dir = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
os.makedirs(out_dir, exist_ok=True)

import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("batch_ground_probe: no CUDA device")

cfg = scans.config(3)
F, N = 512, cfg.points_per_frame
g = cfg.ground
frames = scans.generate(cfg, F, base_seed=0)
dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()
NP = F * N


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


class _DevView:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


result = {"config": 3, "frames": F, "points": NP, "reps": reps}

# (c) the per-frame loop: each call's host time; the messages are gathered outside the timed calls
msgs = [PointCloud2.from_xyzi(f) for f in frames]
loop_out = np.empty((NP, 8), np.float32)
loop_kept = np.zeros(F, np.uint32)
with api.ConesGpu(max_points=N, max_frames=1) as one:
    for f in range(4):
        one.ground_remove(msgs[f], g, copy=False)
    t_loop = []
    for r in range(max(2, reps // 3)):
        total = 0.0
        for f in range(F):
            t = time.perf_counter()
            o, k, _ = one.ground_remove(msgs[f], g, copy=False)
            total += time.perf_counter() - t
            if r == 0:
                loop_out[f * N:(f + 1) * N] = o
                loop_kept[f] = k
        t_loop.append(total * 1e3)
result["loop_ms"] = med(t_loop)
print("per-frame loop", result["loop_ms"], "ms", flush=True)

with api.ConesGpu(max_points=NP, max_frames=F) as h:
    h.set_device_input(dev.data_ptr(), np.full(F, N, np.uint32), keep=dev)
    stream = torch.cuda.ExternalStream(h.lib.cp_stream(h._h))
    host_out = np.empty((NP, 8), np.float32)
    host_out[:] = 0                       # the caller's buffer, its pages faulted in before timing
    kept_h, low_h, cg = np.zeros(F, np.uint32), np.zeros((F, 17), np.float32), to_c_ground(g)
    t_dev, t_ev, t_host = [], [], []
    for r in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        _, kept_d, _ = h.batch_ground_remove(g, host=False)
        e1.record(stream)
        t1 = time.perf_counter()
        e1.synchronize()
        t2 = time.perf_counter()
        st = h.lib.cp_batch_ground_remove(h._h, C.byref(cg), host_out.ctypes.data, NP, kept_h.ctypes.data,
                                          low_h.ctypes.data)
        t3 = time.perf_counter()
        assert st == api.CP_OK
        if r:   # repetition 0 warms up
            t_dev.append((t1 - t0) * 1e3)
            t_ev.append(e0.elapsed_time(e1))
            t_host.append((t3 - t2) * 1e3)
    rows = h.last_rows_loaded()
    assert np.array_equal(kept_d, loop_kept) and np.array_equal(kept_h, loop_kept)
    assert np.array_equal(host_out.view(np.uint32), loop_out.view(np.uint32)), "host output differs from the loop"
    h.batch_ground_remove(g, host=False)
    ptr, n = h.ground_device_output()
    assert n == NP
    got = torch.as_tensor(_DevView(ptr, 32 * n), device="cuda")
    assert torch.equal(got, torch.from_numpy(loop_out.view(np.uint8).reshape(-1)).cuda()), "device output differs"

# the floor: the bytes the call must move over the rate of a device-to-device copy of the output's size
src = torch.empty(32 * NP, dtype=torch.uint8, device="cuda")
dst = torch.empty_like(src)
for _ in range(3):
    dst.copy_(src)
t_cp = []
for _ in range(reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    dst.copy_(src)
    e1.record()
    e1.synchronize()
    t_cp.append(e0.elapsed_time(e1))
copy_rate = 2 * 32 * NP / (med(t_cp) * 1e-3)       # bytes read + written per second
model = {"pass1_read": 16 * NP, "pass2_read": 16 * 32 * rows, "messages_write": 32 * NP}
model_bytes = sum(model.values())
floor_ms = model_bytes / copy_rate * 1e3
result.update({
    "kept_total": int(loop_kept.sum()), "rows_loaded": int(rows), "rows_total": NP // 32,
    "batch_device_ms": med(t_dev), "batch_device_events_ms": med(t_ev), "batch_host_ms": med(t_host),
    "identical": True, "model_bytes": model, "model_gb": model_bytes / 1e9,
    "d2d_copy_tb_s": copy_rate / 1e12, "floor_ms": floor_ms,
    "floor_over_device_events": floor_ms / med(t_ev),
    "loop_over_batch_device": result["loop_ms"] / med(t_dev),
    "loop_over_batch_host": result["loop_ms"] / med(t_host),
})
result["gpu"], result["power_limit"] = card()
print(json.dumps(result))
with open(os.path.join(out_dir, "batch_ground_probe.json"), "w") as f:
    f.write(json.dumps(result) + "\n")
