"""Retrained colour classifiers on the device: `python tools/color_graph_probe.py OUT_DIR [reps] [rounds]`.

Four models on one handle: dam_net (cone_color_kernel), dam_net with one identity RESHAPE (the same arithmetic on
color_graph_kernel), and two larger written models on color_graph_kernel (tests/test_color_graphs.py builds them):
  wide      conv 3x3 SAME 1->32 ReLU, depthwise 3x3 SAME, conv 1x1 32->64 ReLU, max-pool 2x2 SAME, MEAN,
            FC 64->64 ReLU, FC 64->3, softmax
  at_limit  conv 3x3 SAME 1->321 ReLU (the largest activation pair 11 floats under 227 KB), MEAN, FC, softmax
Times with CUDA events on the handle's stream, after warm-up, the models alternated round by round:
  (a) cp_classify_images on 7 911 images (the recorded and synthetic images of tests/golden/cone_images.npz, tiled):
      upload, network, read-back;
  (b) cp_batch_cone_colors after one cp_batch_run of config 3 (512 frames, device-resident input, intensities scaled
      into the range dam_net was trained on).
Medians and spreads (min, max of the per-round medians) per model, the card's name and power limit, and whether the
two dam_net arms agree bit for bit.  Writes one JSON line to OUT_DIR/color_graph_probe.json."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cones_perception_b200 import api, scans  # noqa: E402
from tests.test_color_graphs import Net, arch_at_limit, dam_net_bytes, dam_net_plus_reshape  # noqa: E402

out_dir = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
os.makedirs(out_dir, exist_ok=True)

import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("color_graph_probe: no CUDA device")

GOLD = os.path.join(ROOT, "tests", "golden")
wide = (Net(21).conv(32, 3, 1, "SAME", "RELU", in_scale=0.02).depthwise(1, 3, 1, "SAME", "RELU")
        .conv(64, 1, 1, "VALID", "RELU").pool("MAX_POOL_2D", 2, 2, "SAME").mean().fc(64, "RELU").fc(3).softmax())
MODELS = {"dam_net/cone_color_kernel": dam_net_bytes(), "dam_net/color_graph_kernel": dam_net_plus_reshape(),
          "wide/color_graph_kernel": wide.bytes(), "at_limit/color_graph_kernel": arch_at_limit().bytes()}

z = np.load(os.path.join(GOLD, "cone_images.npz"))
base = np.concatenate([z["real_images"], z["synth_images"]])
imgs = np.ascontiguousarray(np.resize(base, (7911, 15, 12)), np.uint8)
NI = len(imgs)

cfg = scans.config(3)
F, N = 512, cfg.points_per_frame
frames = scans.generate(cfg, F, base_seed=0)
frames[..., 3] = np.clip(frames[..., 3] * 2.5, 0, 255)
dev = torch.from_numpy(frames.reshape(-1, 4)).cuda()

res = {m: {"classify_ms": [], "batch_colors_ms": []} for m in MODELS}
outputs = {}
with api.ConesGpu(max_points=F * N, max_frames=F) as h:
    h.set_device_input(dev.data_ptr(), np.full(F, N, np.uint32), keep=dev)
    stream = torch.cuda.ExternalStream(h.lib.cp_stream(h._h))
    h.color_net_load_tflite(MODELS["dam_net/cone_color_kernel"])
    h.run(cfg.detect, cfg.ground)
    _, off, cl = h.results()
    K = len(cl)
    colors, probs, logits = np.zeros(NI, np.uint8), np.zeros((NI, 3), np.float32), np.zeros((NI, 3), np.float32)
    kcolors, kprobs = np.zeros(K, np.uint8), np.zeros((K, 3), np.float32)
    kflags, kcounts = np.zeros(K, np.uint32), np.zeros(K, np.uint32)

    def classify():
        st = h.lib.cp_classify_images(h._h, imgs.ctypes.data, NI, colors.ctypes.data, probs.ctypes.data,
                                      logits.ctypes.data)
        assert st == 0, h.lib.cp_last_error(h._h)

    def batch():
        st = h.lib.cp_batch_cone_colors(h._h, C.c_float(0.228), C.c_double(0.05), kcolors.ctypes.data,
                                        kprobs.ctypes.data, kflags.ctypes.data, kcounts.ctypes.data, K)
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
        return float(np.median(ms))

    for r in range(rounds):
        for name, model in MODELS.items():
            h.color_net_load_tflite(model)
            res[name]["classify_ms"].append(timed(classify))
            res[name]["batch_colors_ms"].append(timed(batch))
            if r == 0:
                outputs[name] = (colors.copy(), probs.copy(), logits.copy(), kcolors.copy(), kprobs.copy(),
                                 kflags.copy())

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
a, b = outputs["dam_net/cone_color_kernel"], outputs["dam_net/color_graph_kernel"]
same = all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(a, b))
summary = {}
for name, v in res.items():
    summary[name] = {k: {"median_ms": float(np.median(t)), "min_ms": float(np.min(t)), "max_ms": float(np.max(t))}
                     for k, t in v.items()}
line = {"probe": "color_graph", "device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi,
        "images": NI, "batch_frames": F, "batch_clusters": K, "reps": reps, "rounds": rounds,
        "dam_net_arms_bit_identical": same, "models": summary}
print(json.dumps(line))
with open(os.path.join(out_dir, "color_graph_probe.json"), "w") as f:
    f.write(json.dumps(line) + "\n")
