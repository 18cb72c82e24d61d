"""Pass 1 and the per-frame kernel at each CTAs-per-SM cap, then the headline bench alternating two builds.

    python tools/split_sweep.py OLD_LIB [--variants name=ENV=V,ENV=V ...] [--rounds 3] [--out FILE]

OLD_LIB is a libconesgpu.so built from the parent commit; the new build is the tree's own library.  Everything
runs in one process tree so the numbers share one card: the card's name and power limit head the output.
  1. stage timing (CUDA events around each kernel, cp_stage_ms) with one handle open on 512 config-3 frames
     resident in HBM: pass 1 at 1, 2, 3, 4 CTAs per SM, the per-frame kernel at 2, 3, 4 CTAs per SM;
  2. `bench.py --no-sub-records --steps 100`, rounds x (old, new, variants...) in alternation; the CPU baseline is
     cut to one pass over --parity-frames frames, which still yields the oracle parity block of those frames.
Writes nothing into the tree unless --out names a file there."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPS = 20


def stages() -> dict:
    """Child: stage times of the library CONESGPU_LIB (or the tree's) on the bench workload."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    from cones_perception_b200 import api, scans
    cfg = scans.config(3)
    F, N = 512, cfg.points_per_frame
    host = torch.empty((F, N, 4), dtype=torch.float32, pin_memory=True)
    scans.generate(cfg, F, base_seed=0, out=host.numpy())
    dev = host.to("cuda")
    fp = np.full(F, N, np.uint32)

    def timed(env, stage):
        with api.ConesGpu(max_points=F * N, max_frames=F, max_survivors=max(F * N // 8, 1 << 20),
                          max_voxels=max(F * N // 16, 1 << 19), env=env) as h:
            h.set_device_input(dev.data_ptr(), fp, keep=dev)
            h.set_stage_timing(True)
            ms = []
            for i in range(REPS + 3):
                h.run(cfg.detect, cfg.ground)
                h.sync()
                if i >= 3:
                    ms.append(h.stage_ms(stage))
            return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}

    extra = json.loads(os.environ.get("SWEEP_ENV", "{}"))
    out = {"pass1": {}, "frame_kernel": {}}
    for k in (1, 2, 3, 4):
        out["pass1"][str(k)] = timed({**extra, "CONESGPU_K1_CTAS": str(k)}, 0)
    for k in (2, 3, 4):
        out["frame_kernel"][str(k)] = timed({**extra, "CONESGPU_FRAME_CTAS": str(k)}, 4)
    return out


def child(lib, env, *args):
    e = dict(os.environ, **env)
    if lib:
        e["CONESGPU_LIB"] = lib
    r = subprocess.run([sys.executable, *args], cwd=ROOT, env=e, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit(f"{args} failed ({r.returncode}):\n{r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old_lib")
    ap.add_argument("--variants", nargs="*", default=[], help="extra new-build arms: name=ENV=V,ENV=V")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--parity-frames", type=int, default=32, help="frames of the timed batch checked against the oracle")
    ap.add_argument("--out", default=None)
    ap.add_argument("--stages-child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.stages_child:
        print(json.dumps(stages()))
        return
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say(f"card: {smi[0] if smi else 'unknown'}")
    arms = [("old", os.path.abspath(a.old_lib), {}), ("new", None, {})]
    for v in a.variants:
        name, _, spec = v.partition("=")
        arms.append((name, None, dict(kv.split("=", 1) for kv in spec.split(",") if kv)))
    for name, lib, env in arms:
        st = child(lib, {"SWEEP_ENV": json.dumps(env)}, os.path.abspath(__file__), "old", "--stages-child")
        p1 = "  ".join(f"{k}:{v['median_ms']:.4f}" for k, v in st["pass1"].items())
        fk = "  ".join(f"{k}:{v['median_ms']:.4f}" for k, v in st["frame_kernel"].items())
        say(f"stages {name:10s} pass 1 ms by CTAs/SM  {p1}   per-frame kernel ms by CTAs/SM  {fk}")
    res = {name: [] for name, _, _ in arms}
    for r in range(a.rounds):
        for name, lib, env in arms:
            d = child(lib, env, "bench.py", "--no-sub-records", "--steps", str(a.steps), "--cpu-sample-frames",
                      str(a.parity_frames), "--cpu-sample-seconds", "0.01")
            res[name].append(d["ms_per_step"])
            k1 = d.get("roofline", {}).get("kernels", {}).get("ground_sector_min_kernel", {}).get("ms")
            say(f"bench round {r} {name:10s} ms_per_step {d['ms_per_step']:.4f}  pass1 {k1}  "
                f"parity {json.dumps((d.get('cpu_baseline') or {}).get('parity_of_timed_batch'))}")
    for name, v in res.items():
        say(f"bench {name:10s} ms_per_step  mean {sum(v) / len(v):.4f}  min {min(v):.4f}  max {max(v):.4f}  "
            f"runs {' '.join(f'{x:.4f}' for x in v)}")
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
