"""What the node publishes for a whole batch: `python tools/batch_track_probe.py OUT_DIR [reps]`.

Config 3, 512 frames, device-resident input, intensities scaled into the range dam_net was trained on, dam_net loaded,
use_points_buffer on.  After one cp_batch_run, compares two ways to get the published clouds of every frame:
  (a) cp_batch_track                                          one call
  (b) the host path it replaces: cp_batch_results + cp_batch_cone_colors (colour mode), then the C++ ConeTracker
      (host/nodes.hpp) frame by frame through the host library
with colours off and on, as 1 sequence of 512 frames and as 64 sequences of 8.  Both must give identical cones, order
and cloud offsets.  Times are host wall clock around calls that end in a device synchronise (medians of `reps`), plus
the device time of (a) with CUDA events on the handle's stream.  Reports the card's name and power limit.
Writes one JSON line to OUT_DIR/batch_track_probe.json."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cones_perception_b200 import api, scans  # noqa: E402
from cones_perception_b200.build import HOST_LIB  # noqa: E402

out_dir = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
os.makedirs(out_dir, exist_ok=True)

import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("batch_track_probe: no CUDA device")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
cfg = scans.config(3)
F, N = 512, cfg.points_per_frame
d = cfg.detect
frames = scans.generate(cfg, F, base_seed=0)
frames[..., 3] = np.clip(frames[..., 3] * 2.5, 0, 255)
dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()

host = C.CDLL(HOST_LIB)
host.ch_tracker_create.restype = C.c_void_p
host.ch_tracker_create.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double]
host.ch_tracker_destroy.argtypes = [C.c_void_p]
host.ch_tracker_update.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32]
host.ch_tracker_update_answers.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_uint32]
CAP = 4096


def host_path(h, classify, seq_len):
    """cp_batch_results (+ cp_batch_cone_colors) + ConeTracker per frame; returns (xy [n, 2], colour [n], offsets)."""
    _, off, cl = h.results()
    if classify:
        colors, _, flags, _ = h.batch_cone_colors(0.228, d.cone_position_extension_length)
    xs, cs, coff = [], [], [0]
    out = np.zeros((4, CAP, 2), np.float32)
    counts = np.zeros(4, np.uint32)
    t = None
    for f in range(F):
        if f % seq_len == 0:
            if t is not None:
                host.ch_tracker_destroy(t)
            t = host.ch_tracker_create(int(classify), 1, d.cones_matching_dist_theshold,
                                       d.cone_position_extension_length)
        a, b = int(off[f]), int(off[f + 1])
        xy = np.ascontiguousarray(np.stack([cl["x"][a:b], cl["y"][a:b]], 1), np.float32)
        if classify:
            ca, fa = np.ascontiguousarray(colors[a:b]), np.ascontiguousarray(flags[a:b])
            rc = host.ch_tracker_update_answers(t, xy.ctypes.data, b - a, ca.ctypes.data, fa.ctypes.data,
                                                out.ctypes.data, counts.ctypes.data, CAP)
        else:
            rc = host.ch_tracker_update(t, xy.ctypes.data, b - a, -1, out.ctypes.data, counts.ctypes.data, CAP)
        assert rc == 0
        for c in range(4):
            xs.append(out[c, :counts[c]].copy())
            cs.append(np.full(counts[c], c, np.uint32))
            coff.append(coff[-1] + int(counts[c]))
    host.ch_tracker_destroy(t)
    return np.concatenate(xs), np.concatenate(cs), np.array(coff, np.uint32)


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


result = {"config": 3, "frames": F, "reps": reps}
with api.ConesGpu(max_points=F * N, max_frames=F) as h:
    h.color_net_load_tflite(np.load(os.path.join(ROOT, "tests", "golden", "dam_net_model.npz"))["tflite"].tobytes())
    h.set_device_input(dev.data_ptr(), np.full(F, N, np.uint32), keep=dev)
    stream = torch.cuda.ExternalStream(h.lib.cp_stream(h._h))
    h.run(d, cfg.ground)
    _, off, cl = h.results()
    result["clusters"] = int(len(cl))
    for classify in (False, True):
        for seq_len in (F, 8):
            name = f"{'colours' if classify else 'gate'}_{F // seq_len}x{seq_len}"
            seq = np.arange(0, F + 1, seq_len, dtype=np.uint32)
            p = api.track_params(classify, True, d.cones_matching_dist_theshold, d.cone_position_extension_length)
            t_dev, t_ev, t_host = [], [], []
            for r in range(reps + 1):
                h.track_reset()
                h.run(d, cfg.ground)
                h.sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record(stream)
                cones, coff = h.batch_track(p, seq)
                e1.record(stream)
                t1 = time.perf_counter()
                e1.synchronize()
                xy, col, hoff = host_path(h, classify, seq_len)
                t2 = time.perf_counter()
                if r:   # repetition 0 warms up; the outputs are checked on every repetition
                    t_dev.append((t1 - t0) * 1e3)
                    t_ev.append(e0.elapsed_time(e1))
                    t_host.append((t2 - t1) * 1e3)
                same = (np.array_equal(coff, hoff)
                        and np.array_equal(np.stack([cones["x"], cones["y"]], 1).view(np.uint32), xy.view(np.uint32))
                        and np.array_equal(cones["color"], col))
                assert same, f"{name}: cp_batch_track differs from the host path"
            result[name] = {"published": int(len(cones)), "identical": True,
                            "batch_track_ms": med(t_dev), "batch_track_events_ms": med(t_ev),
                            "host_path_ms": med(t_host)}
            print(name, result[name], flush=True)

result["gpu"], result["power_limit"] = card()
print(json.dumps(result))
with open(os.path.join(out_dir, "batch_track_probe.json"), "w") as f:
    f.write(json.dumps(result) + "\n")
