"""Colour classification of a whole batch: `python tools/batch_colors_probe.py OUT_DIR [reps]`.

Config 3, 512 frames, device-resident input (1 GiB: larger than L2), intensities scaled into the range dam_net was
trained on, dam_net loaded.  Times with CUDA events on the handle's stream, after warm-up:
  (a) cp_batch_run + cp_sync
  (b) (a) + cp_batch_cone_colors                        every cluster, one call
  (c) (a) + the per-frame loop it replaces: records back, radial extension on the host, cp_cone_colors per frame
and reports the bytes the colour call moves (a model counted from sizes), its share of the single-read floor
(16 B x all input points at the HBM rate measured in the same run: a device-to-device copy), and the card's name and
power limit.  Writes one JSON line to OUT_DIR/batch_colors_probe.json."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cones_perception_b200 import api, scans  # noqa: E402

out_dir = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
os.makedirs(out_dir, exist_ok=True)

import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("batch_colors_probe: no CUDA device")

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
EXT = 0.05
cfg = scans.config(3)
F, N = 512, cfg.points_per_frame
frames = scans.generate(cfg, F, base_seed=0)
frames[..., 3] = np.clip(frames[..., 3] * 2.5, 0, 255)
dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()


def extend(x, y, ext):
    """src/cone_detection.cpp:276-278 vectorised: float length, float divide, double sum narrowed to float."""
    x, y = x.astype(np.float32), y.astype(np.float32)
    ln = np.sqrt(x.astype(np.float64) ** 2 + y.astype(np.float64) ** 2).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        qx, qy = x / ln, y / ln
    return np.stack([(x.astype(np.float64) + qx.astype(np.float64) * ext).astype(np.float32),
                     (y.astype(np.float64) + qy.astype(np.float64) * ext).astype(np.float32)], 1)


with api.ConesGpu(max_points=F * N, max_frames=F) as h:
    h.color_net_load_tflite(np.load(os.path.join(GOLD, "dam_net_model.npz"))["tflite"].tobytes())
    h.set_device_input(dev.data_ptr(), np.full(F, N, np.uint32), keep=dev)
    stream = torch.cuda.ExternalStream(h.lib.cp_stream(h._h))
    h.run(cfg.detect, cfg.ground)
    _, off, cl = h.results()
    K = len(cl)
    colors, probs = np.zeros(K, np.uint8), np.zeros((K, 3), np.float32)
    flags, counts = np.zeros(K, np.uint32), np.zeros(K, np.uint32)
    # per-frame loop buffers (caller-owned, as a node would hold them)
    lcolors, lflags = np.zeros(K, np.uint8), np.zeros(K, np.uint32)
    lprobs = np.zeros((K, 3), np.float32)
    rec = np.zeros(K, api.CLUSTER_DTYPE)
    offs = np.zeros(F + 1, np.uint32)
    total = C.c_uint64()

    def run():
        h.run(cfg.detect, cfg.ground)
        h.sync()

    def batch():
        run()
        st = h.lib.cp_batch_cone_colors(h._h, C.c_float(0.228), C.c_double(EXT), colors.ctypes.data, probs.ctypes.data,
                                        flags.ctypes.data, counts.ctypes.data, K)
        assert st == 0, h.lib.cp_last_error(h._h)

    def loop():
        run()
        h.lib.cp_batch_results(h._h, None, offs.ctypes.data, rec.ctypes.data, K, C.byref(total))
        centres = extend(rec["x"], rec["y"], EXT)
        for f in range(F):
            a, b = int(offs[f]), int(offs[f + 1])
            if a == b:
                continue
            st = h.lib.cp_cone_colors(h._h, None, f, centres[a:].ctypes.data, b - a, C.c_float(0.228),
                                      lcolors[a:].ctypes.data, lprobs[a:].ctypes.data, lflags[a:].ctypes.data)
            assert st == 0, h.lib.cp_last_error(h._h)

    def timed(fn):
        for _ in range(3):
            fn()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), float(np.min(ms))

    a = timed(run)
    b = timed(batch)
    c = timed(loop)
    batch()
    launches = h.last_launch_count()
    loop()
    same = bool(np.array_equal(colors, lcolors) and np.array_equal(flags, lflags)
                and np.array_equal(probs.view(np.uint32), lprobs.view(np.uint32)))

    # where the colour call's time goes: device time per kernel of one call (torch.profiler, CUDA activity)
    from torch.profiler import ProfilerActivity, profile
    run()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        st = h.lib.cp_batch_cone_colors(h._h, C.c_float(0.228), C.c_double(EXT), colors.ctypes.data, None, None, None, K)
        torch.cuda.synchronize()
    kernel_us = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t:
            kernel_us[ev.key[:60]] = round(float(t), 1)

    # HBM rate: device-to-device copy of 4 GiB (read + write), same process
    src = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(2):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dst.copy_(src)
    e1.record()
    e1.synchronize()
    hbm = 10 * 2 * src.numel() * 4 / (e0.elapsed_time(e1) * 1e-3)
    del src, dst

# one config-2 frame left on the device by cp_detect (a node's duty cycle): the batch call against cp_cone_colors,
# host clock around calls that end in a stream synchronisation, p50 of 200
import time  # noqa: E402

from cones_perception_b200.pointcloud2 import PointCloud2  # noqa: E402

cfg2 = scans.config(2)
f2 = scans.generate(cfg2, 1, base_seed=0)[0]
f2[:, 3] = np.clip(f2[:, 3] * 2.5, 0, 255)
with api.ConesGpu(max_points=len(f2), max_frames=1) as h1:
    h1.color_net_load_tflite(np.load(os.path.join(GOLD, "dam_net_model.npz"))["tflite"].tobytes())
    cl1, _ = h1.detect(PointCloud2.from_xyzi(f2), cfg2.detect, cfg2.ground)
    k1 = len(cl1)
    cen = extend(cl1["x"], cl1["y"], EXT)
    c1, p1, fl1 = np.zeros(k1, np.uint8), np.zeros((k1, 3), np.float32), np.zeros(k1, np.uint32)

    def p50(fn):
        for _ in range(20):
            fn()
        lat = []
        for _ in range(200):
            t = time.perf_counter()
            fn()
            lat.append(1e6 * (time.perf_counter() - t))
        return float(np.percentile(lat, 50))

    single = {
        "clusters": k1,
        "cp_cone_colors_us": p50(lambda: h1.lib.cp_cone_colors(h1._h, None, 0, cen.ctypes.data, k1, C.c_float(0.228),
                                                                c1.ctypes.data, p1.ctypes.data, fl1.ctypes.data)),
        "cp_batch_cone_colors_us": p50(lambda: h1.lib.cp_batch_cone_colors(
            h1._h, C.c_float(0.228), C.c_double(EXT), c1.ctypes.data, p1.ctypes.data, fl1.ctypes.data, None, k1)),
        "batch_launches": int(h1.lib.cp_last_launch_count(h1._h)),
    }

P = int(counts.sum())
n_in = F * N
# bytes of the colour call by kernel, counted from sizes (triples T <= P; P used as the bound):
#   boxes: records + frame offsets read, boxes + frames + counters written; mark: the raw input once (16 B/point),
#   boxes re-read per tile (L1), triples written; sort: prepare + one read and write per live pass of 12 B/triple;
#   gather: matched points re-read, crops written; raster: crops read twice, images written; net: images read.
key_bits = int(np.ceil(np.log2(max(K, 2)))) + int(np.ceil(np.log2(N // 32)))
passes = (key_bits + 7) // 8
parts = {
    "boxes": 16 * K + 4 * (F + 1) + (16 + 4 + 4 + 4) * K,
    "mark_input": 16 * n_in,
    "triples_out": 12 * P,
    "sort": 12 * P * (1 + 2 * passes),
    "gather": 16 * P + 16 * P + 8 * (K + 1),
    "raster": 2 * 16 * P + 180 * K,
    "net": 180 * K + (1 + 4 * 3 + 4) * K,
}
moved = sum(parts.values())
floor_s = 16 * n_in / hbm
extra_s = (b[0] - a[0]) * 1e-3
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:  # noqa: BLE001
    smi = f"unavailable: {e}"
res = {
    "probe": "batch_colors", "config": 3, "frames": F, "points": n_in, "clusters": K, "crop_points": P,
    "colour_launches": launches, "loop_equals_batch": same,
    "a_run_ms": a[0], "b_run_plus_batch_colors_ms": b[0], "c_run_plus_per_frame_loop_ms": c[0],
    "min_ms": {"a": a[1], "b": b[1], "c": c[1]},
    "colour_call_ms": b[0] - a[0], "per_frame_loop_ms": c[0] - a[0],
    "colour_call_bytes_model": moved, "bytes_by_kernel": parts,
    "hbm_copy_GBps": hbm / 1e9, "single_read_floor_ms": floor_s * 1e3,
    "floor_share": floor_s / extra_s if extra_s > 0 else None,
    "colour_call_kernel_us": kernel_us, "single_frame_us": single,
    "device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi, "reps": reps,
}
line = json.dumps(res)
with open(os.path.join(out_dir, "batch_colors_probe.json"), "w") as fh:
    fh.write(line + "\n")
print(line)
