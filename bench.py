#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: points/s (and frames/s, p50 frame
latency) of the cones_perception hot path on 130k-point scans.

    python bench.py --gpus N --steps K --warmup W            # ours (CUDA, libconesgpu.so)
    python bench.py --impl reference --gpus N ...            # the CPU path on the host cores
    python bench.py ... --dump-outputs DIR                   # also writes the last timed step's results as .npy

A step = one pass of the whole hot path (ground removal -> crop -> VoxelGrid -> Euclidean
clustering -> centroids) over one batch of synthetic scans: BASELINE.json config 3, the
64-beam 131 072-point scan with simulation params and ground removal on, FRAMES_PER_GPU
frames per rank (weak scaling: 8 GPUs x 512 = the 4096-frame batch).  One JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cones_perception_b200 import scans  # noqa: E402

METRIC = "points/sec at 130k-pt scans (frames/sec and p50 frame latency in extra keys)"
UNIT = "points/s"
CONE_CAP_PER_FRAME = 64


def env_int(name, default):
    return int(os.environ.get(name, default))


# ------------------------------------------------------------------ clocks sampler
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  The region is short (tens of ms),
    so NVML is polled from a thread every ~2 ms; `nvidia-smi -lms` is the fallback."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm, self.reasons, self.max_sm = [], set(), None
        self._stop = threading.Event()
        self.period = float(os.environ.get("BENCH_CLOCK_PERIOD_S", "0.01"))
        self._thread = None
        self._smi = None

    def _nvml_loop(self):
        import pynvml as nv
        nv.nvmlInit()
        try:
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            while not self._stop.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(self.period)
        finally:
            nv.nvmlShutdown()

    def start(self):
        try:
            import pynvml  # noqa: F401
            # CUDA_VISIBLE_DEVICES may renumber devices; NVML uses physical indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    self.gpu = int(vis.split(",")[self.gpu])
                except (ValueError, IndexError):
                    pass
            self._thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self._thread.start()
            time.sleep(0.02)
        except Exception:
            fields = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                      "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                      "clocks_event_reasons.sw_power_cap")
            try:
                self._smi = subprocess.Popen(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits",
                                              "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                             stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self._smi = None

    def stop(self) -> dict:
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
        elif self._smi is not None:
            time.sleep(0.1)
            self._smi.terminate()
            out, _ = self._smi.communicate(timeout=2)
            for ln in out.splitlines():
                p = [x.strip() for x in ln.split(",")]
                if len(p) >= 7:
                    try:
                        self.sm.append(float(p[1]))
                        self.max_sm = float(p[2])
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                       p[3:7]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ------------------------------------------------------------------ CPU path (oracle)
def cpu_frames_per_sec(frames: np.ndarray, cfg, threads: int, mode_faithful: bool = True, keep: list | None = None):
    """Times the CPU restatement (PCL cost profile) on `frames`; returns (seconds, per-stage ms).
    keep: a list of len(frames) that receives every frame's (clusters, counters) for the parity check."""
    from oracle import oracle as O

    mode = O.PCL_FAITHFUL if mode_faithful else O.CANONICAL
    O.lib()
    stage = {"ground": 0.0, "from_msg": 0.0, "copy_cloud": 0.0, "crop": 0.0, "voxel": 0.0, "cluster": 0.0}
    lock = threading.Lock()

    def work(idx):
        loc = dict.fromkeys(stage, 0.0)
        for i in idx:
            cl, oc, tm = O.detect(O.view_of_xyzi(frames[i]), cfg.detect, cfg.ground, mode)
            if keep is not None:
                keep[i] = (cl, (oc.n_ground_kept, oc.n_cropped, oc.n_voxels, oc.n_components, oc.n_clusters))
            for k in loc:
                loc[k] += getattr(tm, k)
        with lock:
            for k in loc:
                stage[k] += loc[k]

    n = len(frames)
    t0 = time.perf_counter()
    if threads <= 1:
        work(range(n))
    else:
        th = [threading.Thread(target=work, args=(range(t, n, threads),)) for t in range(threads)]
        [t.start() for t in th]
        [t.join() for t in th]
    dt = time.perf_counter() - t0
    return dt, {k: 1e3 * v / n for k, v in stage.items()}


def host_description() -> dict:
    """CPU model, core count and compiler of the CPU arm (SURVEY 8(d): stated in the result file)."""
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.lower().startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    try:
        cc = subprocess.run(["g++", "--version"], capture_output=True, text=True).stdout.splitlines()[0]
    except Exception:
        cc = "g++ (version unknown)"
    return {"cpu_model": model, "host_cores": os.cpu_count(), "compiler": cc,
            "flags": "-O2 -std=c++17 -ffp-contract=off -fno-fast-math (oracle/Makefile)"}


def compare_with_oracle(kept, ctr, k_off, clusters, tol=1e-5):
    """GPU results of a batch against the oracle's (pcl_faithful mode: PCL's own cluster order and summation
    order) for the first len(kept) frames: counters identical, the multiset of (size, min voxel index) per frame
    identical, centroids within `tol` metres (north_star's 1e-5 m).  Raises on any difference."""
    worst = 0.0
    n_cl = 0
    for f, (ocl, oc) in enumerate(kept):
        got = clusters[k_off[f]:k_off[f + 1]]
        names = ("n_ground_kept", "n_cropped", "n_voxels", "n_components", "n_clusters")
        mine = tuple(int(ctr[n][f]) for n in names)
        assert mine == tuple(int(v) for v in oc), f"frame {f}: counters {dict(zip(names, mine))} vs oracle {oc}"
        a = np.sort(got, order=("size", "min_index"))
        b = np.sort(ocl, order=("size", "min_index"))
        assert len(a) == len(b) and np.array_equal(a["size"], b["size"]) and \
            np.array_equal(a["min_index"], b["min_index"]), f"frame {f}: cluster membership differs from the oracle"
        if len(a):
            worst = max(worst, float(np.max(np.abs(a["x"] - b["x"]))), float(np.max(np.abs(a["y"] - b["y"]))))
        n_cl += len(a)
    assert worst <= tol, f"centroids differ from the oracle by {worst} m"
    return {"frames_checked": len(kept), "clusters_checked": n_cl, "max_centroid_diff_m": worst, "tolerance_m": tol,
            "oracle_mode": "pcl_faithful", "what": "counters (G, C, V, components, K) and (size, min index) sets "
            "identical; centroids within tolerance"}


WORKLOAD = ("cfg3: batch of 64-beam 131072-pt scans (simulation params, ground removal on), "
            "{F} frames per GPU, frame-sharded")


def workload_config(F: int, n: int, world: int) -> dict:
    """The part of `config` both arms share (the reference arm is timed on this arm's workload)."""
    return {"workload": WORKLOAD.format(F=F), "frames_per_gpu": F, "points_per_frame": n, "global_frames": world * F}


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return  # only rank 0 measures the CPU path
    cfg = scans.config(3)
    cores = os.cpu_count() or 1
    # a step = the same batch the CUDA arm times per GPU (512 frames: about 0.3 s on 16 host threads)
    sample = args.cpu_step_frames if args.cpu_step_frames > 0 else args.frames_per_gpu
    frames = scans.generate(cfg, sample, base_seed=0)
    n = cfg.points_per_frame
    for _ in range(args.warmup):
        cpu_frames_per_sec(frames[: max(cores, 8)], cfg, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_frames_per_sec(frames, cfg, cores)
    dt = time.perf_counter() - t0
    pts = args.steps * sample * n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": pts, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "frames_per_sec": pts / n,
        "config": {**workload_config(args.frames_per_gpu, n, max(1, env_int("WORLD_SIZE", 1))),
                   "frames_per_step": sample, "parallelism": f"{cores} host threads (rank 0 only)"},
        "cpu_baseline": {"value": pts, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} frames/step of the same scans, oracle pcl_faithful mode, "
                                   f"g++ -O2, frame-parallel over {cores} threads",
                         "host": host_description()},
        "e2e": {"value": pts, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ ours
DUMP_BYTES_MAX = 64_000_000
NPY_HEADER_MAX = 4096            # an .npy header of a 1-D array is 128 bytes; counted generously


def dump_outputs(out_dir: str, ctr, k_off, clusters, prefix: str = "", budget: int = DUMP_BYTES_MAX) -> None:
    """Writes one step's results, what ConesGpu.results() hands a caller, as float .npy files so that two builds
    can be compared output for output: per-frame counters, cluster offsets and the cluster records field by field.
    Integers are stored as float64 (exact below 2**53).  Cluster lists larger than the byte budget are cut to a
    seeded random subset of records, whose indices are stored beside them.  `budget` bounds the files' total size,
    headers included."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {f"counters_{n}": ctr[n].astype(np.float64) for n in ctr.dtype.names}
    arrays["cluster_offsets"] = k_off.astype(np.float64)
    fixed = sum(a.nbytes for a in arrays.values()) + (len(arrays) + 5) * NPY_HEADER_MAX
    per_record = 4 + 4 + 8 + 8 + 8          # x, y (float32) + size, min_index, sample index (float64)
    keep = max(0, (budget - fixed) // per_record)
    if len(clusters) > keep:
        idx = np.sort(np.random.default_rng(0).choice(len(clusters), keep, replace=False))
        clusters = clusters[idx]
        arrays["clusters_sample_index"] = idx.astype(np.float64)
    for n in ("x", "y"):
        arrays[f"clusters_{n}"] = np.ascontiguousarray(clusters[n], np.float32)
    for n in ("size", "min_index"):
        arrays[f"clusters_{n}"] = clusters[n].astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a)


class _DevArray:
    """Zero-copy torch view of a raw device pointer (result buffers of the library)."""

    def __init__(self, ptr: int, shape, typestr="<i4"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False),
                                         "version": 2}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from cones_perception_b200 import api
    from cones_perception_b200.pointcloud2 import PointCloud2, make_view, CCloudView
    from cones_perception_b200.sharding import gather_cone_lists, pack_words, setup_peer_gather

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # exactly one line may reach stdout (the JSON): park stdout on stderr while libraries (NCCL
    # version banners, torchrun notices) are chatty, print the line on the real stdout at the end
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libconesgpu has no CPU fallback")
    # Which GPU a rank drives.  On HGX boards GPUs 0..3 and 4..7 hang off different host uplinks (measured here:
    # four ranks on GPUs 0-3 share 115 GB/s of host->device bandwidth, profiles/r02_h2d/); when the job uses fewer
    # GPUs than the box shows, ranks are dealt alternately to the two halves so they do not crowd one uplink.
    ndev = torch.cuda.device_count()
    dev_index = local
    if 1 < world < ndev and ndev % 2 == 0 and os.environ.get("BENCH_SPREAD", "1") != "0":
        perm = [x for pair in zip(range(ndev // 2), range(ndev // 2, ndev)) for x in pair]
        dev_index = perm[local]
    torch.cuda.set_device(dev_index)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev_index))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_obj(v):
        if world == 1:
            return [v]
        out = [None] * world
        dist.all_gather_object(out, v)
        return out

    # ---- host placement, then the box's raw host->device ceiling (both BEFORE the pinned batch is allocated).
    # Ranks look for their CPU group one after the other (the placement probes must not disturb each other);
    # the ceiling is then measured with every rank copying at the same time.
    from cones_perception_b200 import placement
    bind = {"how": "single rank: not bound"}
    if world > 1 and os.environ.get("BENCH_BIND", "1") != "0":
        for r in range(world):
            if r == rank:
                try:
                    bind = placement.bind_rank(dev_index)
                except Exception as e:            # never let placement stop the measurement
                    bind = {"how": f"failed ({type(e).__name__}: {e})"}
            barrier()
    probe = placement.h2d_probe(dev_index, 1 << 30, 6, barrier)
    probes = gather_obj({"GBps": probe["GBps"], "bind": bind, "pages_by_node": probe["pages_by_node"],
                         "device": dev_index})

    cfg = scans.config(3)
    F, N = args.frames_per_gpu, cfg.points_per_frame
    d, g = cfg.detect, cfg.ground

    # ---- synthetic input: this rank's contiguous shard of the global batch, pinned
    host = torch.empty((F, N, 4), dtype=torch.float32, pin_memory=True)
    hnp = host.numpy()
    scans.generate(cfg, F, base_seed=rank * F, out=hnp)
    dev = host.to("cuda", non_blocking=False)

    gpu = api.ConesGpu(max_points=F * N, max_frames=F, device=dev_index, max_survivors=max(F * N // 8, 1 << 20),
                       max_voxels=max(F * N // 16, 1 << 19))
    ext = torch.cuda.ExternalStream(gpu.stream(), device=torch.device("cuda", dev_index))
    frame_points = np.full(F, N, dtype=np.uint32)
    gpu.set_device_input(dev.data_ptr(), frame_points, keep=dev)
    cone_cap = F * CONE_CAP_PER_FRAME
    # Several batches in flight (--lanes, default 4): consecutive steps go round the handles (one stream and one
    # set of intermediates each), so the latency-bound per-frame kernel of one batch overlaps the HBM-bound first
    # pass of another.  Every step still runs the whole path on the whole batch.
    lanes = [gpu]
    for _ in range(1, max(1, args.lanes)):
        h2 = api.ConesGpu(max_points=F * N, max_frames=F, device=dev_index, max_survivors=max(F * N // 8, 1 << 20),
                          max_voxels=max(F * N // 16, 1 << 19))
        h2.set_device_input(dev.data_ptr(), frame_points, keep=dev)
        lanes.append(h2)
    exts = [torch.cuda.ExternalStream(h.stream(), device=torch.device("cuda", dev_index)) for h in lanes]

    # result path when N > 1: the rank's packed cone list (offsets + records, one device block)
    # is copied to a staging buffer on the compute stream and gathered to rank 0 with ONE
    # all_gather on a side stream, overlapping the next step's kernels (KB-scale, latency-bound)
    words = pack_words(F, cone_cap)
    # preferred: peer-memory publish inside the library (no collective on the step path);
    # BENCH_GATHER=nccl keeps the all_gather variant, BENCH_GATHER=0 disables the result path
    gather_mode = os.environ.get("BENCH_GATHER", "peer") if world > 1 else "none"
    if gather_mode == "peer":
        try:
            for h in lanes:
                setup_peer_gather(h, rank, world, F, cone_cap)
        except Exception as e:  # CUDA IPC unavailable: fall back to the collective
            print(f"[bench] peer gather unavailable ({e}); using NCCL all_gather", file=sys.stderr)
            gather_mode = "nccl"
        flags = torch.tensor([1 if gather_mode == "peer" else 0], device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        if int(flags.item()) == 0:
            gather_mode = "nccl"
    if gather_mode == "nccl":
        lanes, exts = lanes[:1], exts[:1]      # the collective fallback keeps one batch in flight
    # high priority: the collective's few CTAs get SM slots ahead of the next step's grid-filling kernels
    comm = torch.cuda.Stream(priority=-1) if world > 1 else None
    stage = [torch.empty(words, dtype=torch.int32, device="cuda") for _ in range(2)] if world > 1 else None
    stage_free = [None, None]
    gathered = [None]
    step_no = [0]

    src_view = [None]
    ready = [torch.cuda.Event(), torch.cuda.Event()] if world > 1 else None
    freed = [torch.cuda.Event(), torch.cuda.Event()] if world > 1 else None

    lane_no = [0]

    def step_device():
        lanes[lane_no[0] % len(lanes)].run(d, g)
        lane_no[0] += 1
        if gather_mode == "nccl":
            i = step_no[0] & 1
            step_no[0] += 1
            if src_view[0] is None:                    # the library's result block has a fixed address
                _, d_off, _ = gpu.device_results()
                src_view[0] = torch.as_tensor(_DevArray(d_off, (words,)), device="cuda")
            if stage_free[i] is not None:
                ext.wait_event(freed[i])               # the gather that last used this buffer is done
            with torch.cuda.stream(ext):
                stage[i].copy_(src_view[0])
            ready[i].record(ext)
            comm.wait_event(ready[i])
            with torch.cuda.stream(comm):
                gathered[0] = gather_cone_lists(stage[i])
                freed[i].record(comm)
                stage_free[i] = True

    def drain():
        if world > 1 and comm is not None:
            ext.wait_stream(comm)
        for e in exts[1:]:
            ext.wait_stream(e)                      # lane 0's stream waits for the other lane

    for _ in range(max(args.warmup, 3) * len(lanes)):
        step_device()
    drain()
    for h in lanes:
        h.sync()
    torch.cuda.synchronize()
    lane_no[0] = 0
    ctr, k_off, clusters = gpu.results()
    launches_per_step = gpu.last_launch_count()

    # ---- timed region: K steps, inputs resident in HBM (1 GiB per rank > 126 MB L2)
    sampler = ClockSampler(dev_index)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for e in exts[1:]:
        e.wait_event(e0)                            # no lane starts before the start event
    for _ in range(args.steps):
        step_device()
    drain()
    e1.record(ext)
    barrier()
    gpu.sync()
    for h in lanes:
        h.sync()
    if args.dump_outputs:
        # the handle that ran the last timed step still holds its results (nothing has run on it since); every
        # rank writes its own, and together they stay within the byte budget
        dump_outputs(args.dump_outputs, *lanes[(args.steps - 1) % len(lanes)].results(),
                     prefix=f"rank{rank}_" if world > 1 else "", budget=DUMP_BYTES_MAX // world)
    if gather_mode == "peer" and rank == 0:
        last = lanes[(args.steps - 1) % len(lanes)]
        seq = last.gather_seq()
        last.gather_wait(seq)
        gathered[0] = torch.from_numpy(last.gather_read(seq, world, words))
    # ---- result path check, EVERY rank's block: each rank hashes the results it read itself (cp_batch_results),
    # the hashes travel over NCCL, and rank 0 compares them with what every peer published into its memory.
    # A second run with a different min_cluster_size changes the cone lists, so a stale double-buffer slot or a
    # misrouted rank cannot pass by showing an older, identical-looking block.
    import hashlib
    from dataclasses import replace
    from cones_perception_b200.sharding import offset_words

    def block_hash(off, recs):
        k = int(off[-1])
        return hashlib.sha256(np.ascontiguousarray(off, np.uint32).tobytes() +
                              np.ascontiguousarray(recs[:k]).view(np.uint32).tobytes()).hexdigest()

    def check_gather(g_np, hashes, what):
        gw = np.ascontiguousarray(g_np).view(np.uint32).reshape(world, -1)
        for r in range(world):
            off = gw[r, :F + 1]
            recs = gw[r, offset_words(F):].reshape(-1, 4)
            assert block_hash(off, recs) == hashes[r], f"{what}: rank {r}'s published cone list differs from its own"

    gather_check = None
    if world > 1:
        my_hash = block_hash(k_off, clusters)
        hashes = gather_obj(my_hash)
        if rank == 0 and gathered[0] is not None:
            check_gather(gathered[0].cpu().numpy(), hashes, "timed run")
        # second run, different parameters -> different lists, fresh sequence number
        d_alt = replace(d, min_cluster_size=d.min_cluster_size + 1)
        h_alt = lanes[args.steps % len(lanes)]
        barrier()
        h_alt.run(d_alt, g)
        h_alt.sync()
        _, off_alt, cl_alt = h_alt.results()
        alt_hashes = gather_obj(block_hash(off_alt, cl_alt))
        if gather_mode == "peer" and rank == 0:
            seq = h_alt.gather_seq()
            h_alt.gather_wait(seq)
            check_gather(h_alt.gather_read(seq, world, words), alt_hashes, "changed-parameter run")
        elif gather_mode == "nccl":
            stage[0].copy_(torch.as_tensor(_DevArray(h_alt.device_results()[1], (words,)), device="cuda"))
            got = gather_cone_lists(stage[0])
            if rank == 0:
                check_gather(got.cpu().numpy(), alt_hashes, "changed-parameter run")
        gather_check = {"ranks_checked": world, "runs_checked": 2 if gathered[0] is not None or rank else 1,
                        "changed_run_differs": bool(alt_hashes[0] != hashes[0]),
                        "how": "sha256 of every rank's own cp_batch_results vs the block it published on rank 0"}
        barrier()
        h_alt.run(d, g)           # leave the handle (and its replay graph) on the benchmark parameters
        h_alt.sync()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = world * F * N * args.steps / (ms_total * 1e-3)

    # ---- per-kernel roofline pass (events around each streaming kernel, same workload)
    gpu.set_stage_timing(True)
    k1, k2, kf, kc = [], [], [], []
    k2_name = ["keep_mask_kernel"]
    for _ in range(min(args.steps, 10)):
        gpu.run(d, g)
        gpu.sync()
        try:
            kc.append(gpu.stage_ms(3))          # front_cluster_kernel: one HBM pass, points stashed in smem
        except api.ConesGpuError:
            try:
                kf.append(gpu.stage_ms(2))      # front_fused_kernel: both passes in one launch, pass 2 from L2
            except api.ConesGpuError:
                k1.append(gpu.stage_ms(0))
                try:
                    k2.append(gpu.stage_ms(1))
                except api.ConesGpuError:
                    k2.append(gpu.stage_ms(4))      # pass 2 runs inside the per-frame kernel
                    k2_name[0] = "frame_backend_kernel"
    gpu.set_stage_timing(False)
    C_tot, V_tot, K_tot = int(ctr["n_cropped"].sum()), int(ctr["n_voxels"].sum()), int(ctr["n_clusters"].sum())
    mask_bytes = F * N // 8
    kernels = {}
    if kc:
        # one pass over HBM: the compulsory traffic is 16 B/pt + the keep mask; SURVEY 8(d)'s two-pass figure
        # (32 B/pt) is what the same work costs without the shared-memory stash and is reported beside it
        kc_ms = float(np.mean(kc))
        bytes_kc = 16 * F * N + mask_bytes
        kernels["front_cluster_kernel"] = {"ms": kc_ms, "GBps": bytes_kc / (kc_ms * 1e-3) / 1e9,
                                           "two_pass_equivalent_GBps": (32 * F * N + mask_bytes) / (kc_ms * 1e-3) / 1e9}
        dom = ("front_cluster_kernel", kc_ms, bytes_kc)
    elif kf:
        # algorithmic bytes per SURVEY 8(d): both passes read the scan (16 B/pt each) + the keep mask;
        # the HBM interface is crossed once (pass 2 re-reads from L2), reported as the single-read figure
        kf_ms = float(np.mean(kf))
        bytes_kf = 32 * F * N + mask_bytes
        kernels["front_fused_kernel"] = {"ms": kf_ms, "GBps": bytes_kf / (kf_ms * 1e-3) / 1e9,
                                         "single_read_GBps": (16 * F * N + mask_bytes) / (kf_ms * 1e-3) / 1e9}
        dom = ("front_fused_kernel", kf_ms, bytes_kf)
    else:
        k1_ms, k2_ms = float(np.mean(k1)), float(np.mean(k2))
        # pass 1 reads every point and writes one row-maximum per 32 points; pass 2 reads the row maxima,
        # only the rows that are not entirely below every ground threshold (counted by the library), and
        # writes the keep mask.  Both figures are the bytes the kernels must move, measured per launch.
        rows_total = F * N // 32
        rows_read = gpu.last_rows_loaded()
        bytes_k1 = 16 * F * N + 4 * rows_total
        bytes_k2 = 512 * rows_read + 4 * rows_total + mask_bytes
        kernels["ground_sector_min_kernel"] = {"ms": k1_ms, "GBps": bytes_k1 / (k1_ms * 1e-3) / 1e9}
        if k2_name[0] == "frame_backend_kernel":
            # pass 2 lives in the per-frame kernel: row maxima + live rows in, survivors stay in shared memory
            # (no keep mask is written), cone records out
            bytes_k2 = 512 * rows_read + 4 * rows_total + 16 * int(ctr["n_clusters"].sum())
        kernels[k2_name[0]] = {"ms": k2_ms, "GBps": bytes_k2 / (k2_ms * 1e-3) / 1e9,
                               "rows_read_fraction": rows_read / rows_total,
                               "what": "pass 2 (ground verdicts + crop) of the live rows" +
                                       (", VoxelGrid, clustering, centroids: one CTA per frame"
                                        if k2_name[0] == "frame_backend_kernel" else "")}
        dom = ("ground_sector_min_kernel", k1_ms, bytes_k1) if k1_ms >= k2_ms else (k2_name[0], k2_ms, bytes_k2)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    achieved = dom[2] / (dom[1] * 1e-3) / 1e9
    key_bits = int(ctr["key_bits"].max())
    P = (key_bits + 7) // 8
    b_alg_step = 32 * F * N + (72 + 16 * P) * C_tot + 104 * V_tot + 16 * K_tot
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(dom[0])
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "frac_note": "the peak is the driver-measured torch copy (read + write) bandwidth; this kernel only "
                             "reads (16 B/point + 4 B written per 32 points), and a read-only stream runs slightly above "
                             "the copy figure, so frac can exceed 1; ncu DRAM bytes (traffic) equal the algorithmic bytes",
                "algorithmic_bytes_per_launch": dom[2], "kernel_ms": dom[1],
                "kernels": kernels}
    # whole-step fractions of the measured peak.  bytes moved = what the step's kernels actually read and write
    # (library counters: every point once in pass 1, the row maxima out and in, only the rows pass 2 could not
    # skip, the cone records); single read = the strict bound of one pass over the scan plus the results.
    # SURVEY 8(d)'s B_alg charges two full passes (32 B/point); it is listed for reference only, a step that
    # skips provably-ground rows moves less than that.
    step_s = ms_total * 1e-3 / args.steps
    rows_total = F * N // 32
    rows_read_step = gpu.last_rows_loaded()
    moved = 16 * F * N + 8 * rows_total + 512 * rows_read_step + 16 * K_tot
    single = 16 * F * N + 16 * K_tot
    roofline.update({
        "step_bytes_moved": moved, "step_frac_bytes_moved": moved / step_s / 1e9 / peak,
        "step_bytes_single_read": single, "step_frac_single_read": single / step_s / 1e9 / peak,
        "survey_b_alg_bytes_per_step": b_alg_step,
        "step_note": "fractions of the measured HBM peak over the whole step (all kernels, all batches in flight); "
                     "profiles/traffic.json holds the ncu DRAM sum of the same step"})

    # ---- end to end through the C ABI with HOST buffers (page-locked): H2D + pipeline + D2H
    from cones_perception_b200.params import to_c_detect, to_c_ground
    import ctypes as C
    cd, cg = to_c_detect(d), to_c_ground(g)
    lib = gpu.lib

    def ck(h, st):
        if st != 0:
            raise RuntimeError(lib.cp_last_error(h._h).decode())

    class E2E:
        """One rank's end-to-end loop over `frames` host clouds (numpy [Fx, N, 4] in page-locked memory)."""

        def __init__(self, handles, frames_np, expect_clusters):
            self.handles, self.Fx = handles, len(frames_np)
            self.msgs = [PointCloud2.from_xyzi(frames_np[f]) for f in range(self.Fx)]
            self.views = (CCloudView * self.Fx)(*[make_view(m, True) for m in self.msgs])
            self.cap = self.Fx * CONE_CAP_PER_FRAME
            self.o_ctr = np.zeros(self.Fx, dtype=api.COUNTER_DTYPE)
            self.o_off = np.zeros(self.Fx + 1, dtype=np.uint32)
            self.o_cl = np.zeros(self.cap, dtype=api.CLUSTER_DTYPE)
            self.total = C.c_uint64()
            self.expect = expect_clusters

        def submit(self, h):        # H2D of the batch (page-locked -> device) + the whole pipeline, asynchronous
            ck(h, lib.cp_batch_set_host_input(h._h, self.views, self.Fx))
            ck(h, lib.cp_batch_run(h._h, C.byref(cd), C.byref(cg)))

        def collect(self, h):       # D2H of counters, offsets and the cone list of the handle's batch
            ck(h, lib.cp_batch_results(h._h, self.o_ctr.ctypes.data, self.o_off.ctypes.data, self.o_cl.ctypes.data,
                                       self.cap, C.byref(self.total)))

        def run(self, n):
            # with two handles, the copy of batch i+1 overlaps the kernels and the result read of batch i
            pending = []
            for i in range(n):
                h = self.handles[i % len(self.handles)]
                if len(pending) == len(self.handles):
                    self.collect(pending.pop(0))
                self.submit(h)
                pending.append(h)
            while pending:
                self.collect(pending.pop(0))

        def timed(self, steps, global_frames):
            self.run(2 * len(self.handles))
            barrier()
            t0 = time.perf_counter()
            self.run(steps)
            self.local_s = time.perf_counter() - t0          # this rank's own loop, before it waits for the others
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], device="cuda")
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            k = len(self.expect)
            assert self.total.value == k and np.array_equal(self.o_cl[:k].view(np.uint32), self.expect.view(np.uint32)), \
                "host-input and device-input runs disagree"
            return global_frames * N * steps / float(dt.item())

    e2e_steps = max(4, min(args.steps, 10))
    even = E2E(lanes, hnp, clusters)
    e2e_pinned = even.timed(e2e_steps, world * F)
    clocks = sampler.stop() if rank == 0 else None   # sampled across both timed regions (resident + e2e)
    # the same batch in write-combined page-locked memory (cp_pinned_alloc(.., write_combined = 1)): the DMA reads
    # it without snooping CPU caches.  Same public call; reported beside the default.
    e2e_wc = None
    if os.environ.get("BENCH_WC", "1") != "0":
        try:
            wc = api.PinnedBuffer(F * N * 16, device=dev_index, write_combined=True)
            wnp = wc.array.view(np.float32).reshape(F, N, 4)
            np.copyto(wnp, hnp)
            e2e_wc = E2E(lanes, wnp, clusters).timed(e2e_steps, world * F)
            del wnp
            wc.close()
        except Exception as e:
            print(f"[bench] write-combined variant skipped: {e}", file=sys.stderr)
            e2e_wc = None
    flags = torch.tensor([1.0 if e2e_wc is not None else 0.0], device="cuda")
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if float(flags.item()) == 0.0:
        e2e_wc = None
    # Shards weighted by each rank's measured host link: the step ends with the slowest rank, so on a box whose
    # GPUs do not all get the same host->device rate (shared PCIe uplinks, one socket's memory) equal shards leave
    # the faster links idle.  Same global batch (world x F frames, contiguous blocks), block sizes proportional to
    # the probe's per-rank GB/s.
    probe_rates = [p_["GBps"] for p_ in probes]
    probe_total = float(sum(probe_rates))
    e2e_weighted, shard_sizes, shard_trail = None, None, []
    force_w = os.environ.get("BENCH_WEIGHTED") == "force"          # (testing the path on a box with equal links)
    if world > 1 and (max(probe_rates) > 1.05 * min(probe_rates) or force_w) and \
            os.environ.get("BENCH_WEIGHTED", "1") != "0":
        tot = world * F

        def split(weights):
            wsum = float(sum(weights))
            raw = [tot * w_ / wsum for w_ in weights]
            sizes = [max(1, min(2 * F, int(x))) for x in raw]
            order = sorted(range(world), key=lambda i: raw[i] - int(raw[i]), reverse=True)
            i = 0
            while sum(sizes) < tot:                    # hand the remainder to the largest fractional parts
                if sizes[order[i % world]] < 2 * F:
                    sizes[order[i % world]] += 1
                i += 1
            return sizes

        weights = [r_ * (1.0 + 0.2 * i_) for i_, r_ in enumerate(probe_rates)] if force_w else list(probe_rates)
        for attempt in range(5):
            sizes = split(weights)
            if shard_trail and sizes == shard_trail[-1]["frames"]:
                break
            Fw, first = sizes[rank], sum(sizes[:rank])
            hw_t = torch.empty((Fw, N, 4), dtype=torch.float32, pin_memory=True)
            scans.generate(cfg, Fw, base_seed=first, out=hw_t.numpy())
            dw = hw_t.to("cuda")
            hws = [api.ConesGpu(max_points=Fw * N, max_frames=Fw, device=dev_index,
                                max_survivors=max(Fw * N // 8, 1 << 20), max_voxels=max(Fw * N // 16, 1 << 19))
                   for _ in lanes]
            fpw = np.full(Fw, N, dtype=np.uint32)
            hws[0].set_device_input(dw.data_ptr(), fpw, keep=dw)       # the expected cones: a device-input run
            hws[0].run(d, g)
            _, _, cl_w = hws[0].results()
            run_w = E2E(hws, hw_t.numpy(), cl_w)
            val = run_w.timed(e2e_steps, tot)
            times = gather_obj(run_w.local_s)
            shard_trail.append({"frames": sizes, "value": val, "rank_seconds": times})
            for h in hws:
                h.close()
            del dw, hw_t, run_w
            if e2e_weighted is None or val > e2e_weighted:
                e2e_weighted, shard_sizes = val, sizes
            # next split: frames in proportion to what each rank actually moved per second in this run (the links
            # share upstream bandwidth, so the rates under the new split differ a little from the probe's)
            weights = [sz / max(t_, 1e-9) for sz, t_ in zip(sizes, times)]
            if max(times) < 1.03 * min(times):
                break
    e2e_val = max(e2e_pinned, e2e_wc or 0.0, e2e_weighted or 0.0)
    which = "weighted_shards" if e2e_val == e2e_weighted else ("write_combined" if e2e_val == e2e_wc else "pinned")
    d2h = int(even.o_ctr.nbytes + even.o_off.nbytes + K_tot * 16 + 64)
    e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(F * N * 16), "d2h_bytes_per_step": d2h,
           "frames_per_sec": e2e_val / N, "steps": e2e_steps,
           "variant": which,
           "variants": {"pinned": e2e_pinned, "write_combined": e2e_wc, "weighted_shards": e2e_weighted},
           "weighted_shard_frames": shard_sizes, "weighted_shard_attempts": shard_trail,
           "h2d_GBps": e2e_val * 16 / 1e9,
           "h2d_probe_GBps": {"per_rank": probe_rates, "aggregate": probe_total,
                              "equal_shard_ceiling": world * min(probe_rates),
                              "how": "every rank at the same time: 6 x 1 GiB pinned cudaMemcpyAsync, CUDA events "
                                     "(cones_perception_b200/placement.py h2d_probe), after rank placement; with "
                                     "equal shards the step ends with the slowest link (world x min)"},
           "frac_of_probe": e2e_val * 16 / 1e9 / probe_total if probe_total > 0 else None,
           "frac_of_equal_shard_ceiling": e2e_pinned * 16 / 1e9 / (world * min(probe_rates)),
           "placement": [p_["bind"] for p_ in probes], "devices": [p_["device"] for p_ in probes],
           "h2d_bytes_per_step_note": "per rank with equal shards; weighted shards move the same global bytes",
           "timer": "host wall clock around cp_batch_set_host_input + cp_batch_run + cp_batch_results per step "
                    f"(page-locked host clouds), {len(lanes)} batch(es) in flight"}

    # ---- sub-records: the same step under other conditions (all inside the default command)
    subs = {}
    dev_t = torch.device("cuda", dev_index)
    rows_total = F * N // 32

    def new_handle(frames, env=None):
        h = api.ConesGpu(max_points=frames * N, max_frames=frames, device=dev_index,
                         max_survivors=max(frames * N // 8, 1 << 20), max_voxels=max(frames * N // 16, 1 << 19),
                         env=env)
        return h

    def timed_run(handles, n_steps, dp=d, gp=g):
        """Device-resident ms/step over n_steps, handles alternating; CUDA events; max over ranks."""
        sts = [torch.cuda.ExternalStream(h.stream(), device=dev_t) for h in handles]
        for i in range(3 * len(handles)):
            handles[i % len(handles)].run(dp, gp)
        for h in handles:
            h.sync()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(sts[0])
        for s_ in sts[1:]:
            s_.wait_event(a)
        for i in range(n_steps):
            handles[i % len(handles)].run(dp, gp)
        for s_ in sts[1:]:
            sts[0].wait_stream(s_)
        b.record(sts[0])
        barrier()
        for h in handles:
            h.sync()
        t = torch.tensor([a.elapsed_time(b)], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n_steps

    if args.sub_records:
        sub_steps = max(4, min(args.steps, 20))
        # (1) the exact row skip switched off: pass 2 reads every row
        hs = [new_handle(F, env={"CONESGPU_ROWSKIP": "0"}) for _ in lanes]
        for h in hs:
            h.set_device_input(dev.data_ptr(), frame_points, keep=dev)
        ms_ = timed_run(hs, sub_steps)
        _, off_, cl_ = hs[0].results()
        assert np.array_equal(cl_.view(np.uint32), clusters.view(np.uint32)), "row skip changes the result"
        subs["rowskip_off"] = {"ms_per_step": ms_, "value": world * F * N / (ms_ * 1e-3), "unit": UNIT,
                               "rows_read_fraction": hs[0].last_rows_loaded() / rows_total,
                               "what": "same step with CONESGPU_ROWSKIP=0 (pass 2 reads the whole scan again)"}
        for h in hs:
            h.close()
        # (2) the same scans in firing order (azimuth-major: a 32-point row mixes 32 beams), as an unorganised
        # Velodyne driver publishes them; results checked against the oracle on the permuted clouds
        dev_az = dev.view(F, cfg.beams, cfg.az * cfg.sweeps, 4).transpose(1, 2).contiguous()
        for h in lanes:
            h.set_device_input(dev_az.data_ptr(), frame_points, keep=dev_az)
        ms_ = timed_run(lanes, sub_steps)
        ctr_a, off_a, cl_a = lanes[0].results()
        az = {"ms_per_step": ms_, "value": world * F * N / (ms_ * 1e-3), "unit": UNIT,
              "rows_read_fraction": lanes[0].last_rows_loaded() / rows_total,
              "clusters_per_step": int(off_a[-1]),
              "what": "same scans permuted from ring-major to firing order (azimuth-major)"}
        if rank == 0 and args.cpu_sample_frames > 0:
            from oracle import oracle as O
            nchk = min(8, F)
            az_host = dev_az[:nchk].cpu().numpy()
            kept = []
            for f in range(nchk):
                ocl, oc, _ = O.detect(O.view_of_xyzi(az_host[f]), d, g, O.CANONICAL)
                kept.append((ocl, (oc.n_ground_kept, oc.n_cropped, oc.n_voxels, oc.n_components, oc.n_clusters)))
                got = cl_a[off_a[f]:off_a[f + 1]]
                assert np.array_equal(got.view(np.uint32), ocl.view(np.uint32)), f"azimuth-major frame {f} differs"
            compare_with_oracle(kept, ctr_a, off_a, cl_a)
            az["oracle_checked_frames"] = nchk
        subs["azimuth_major"] = az
        for h in lanes:
            h.set_device_input(dev.data_ptr(), frame_points, keep=dev)
        del dev_az
        # (3) BASELINE.json config 3 as worded: ONE batch of 4096 scans, sharded over the GPUs (strong scaling)
        G_FR = args.strong_frames
        Fs = G_FR // world
        if Fs == F:
            subs["strong_4096"] = {"frames_per_gpu": Fs, "global_frames": G_FR, "ms_per_step": ms_total / args.steps,
                                   "value": value, "unit": UNIT, "scaling": "strong",
                                   "what": "identical to the headline at this N (4096 / N = frames per GPU)"}
        elif Fs > 0:
            dev_s = torch.empty((Fs, N, 4), dtype=torch.float32, device=dev_t)
            for c0 in range(0, Fs, F):
                nc = min(F, Fs - c0)
                scans.generate(cfg, nc, base_seed=rank * Fs + c0, out=hnp[:nc])
                dev_s[c0:c0 + nc].copy_(host[:nc])
            scans.generate(cfg, F, base_seed=rank * F, out=hnp)        # the pinned batch back to the headline's frames
            fp_s = np.full(Fs, N, dtype=np.uint32)
            hs = [new_handle(Fs) for _ in lanes]
            for h in hs:
                h.set_device_input(dev_s.data_ptr(), fp_s, keep=dev_s)
            ms_ = timed_run(hs, sub_steps)
            ctr_s, off_s, cl_s = hs[0].results()
            if rank == 0:      # rank 0's shard starts with the headline's frames (same seeds): same cones
                nf = min(F, Fs)
                assert np.array_equal(cl_s[:off_s[nf]].view(np.uint32), clusters[:k_off[nf]].view(np.uint32)), \
                    "the 4096-frame batch disagrees with the headline batch on their common frames"
            subs["strong_4096"] = {"frames_per_gpu": Fs, "global_frames": Fs * world, "ms_per_step": ms_,
                                   "value": world * Fs * N / (ms_ * 1e-3), "unit": UNIT,
                                   "frames_per_sec": world * Fs / (ms_ * 1e-3), "scaling": "strong",
                                   "clusters_per_step_rank0": int(off_s[-1]),
                                   "input_GB_per_gpu": Fs * N * 16 / 1e9,
                                   "what": f"one batch of {Fs * world} scans, {Fs} per GPU, device-resident, "
                                           f"{len(hs)} batches in flight"}
            for h in hs:
                h.close()
            del dev_s
        # (4) BASELINE.json configs 4 and 5 (N = 1 only): dense 2.6 M-point frames / adversarial clustering
        if world == 1:
            for idx in (4, 5):
                cfgx = scans.config(idx)
                rec = {}
                for Fx in (1, 8):
                    fr = scans.generate_config5(Fx, 0) if idx == 5 else scans.generate(cfgx, Fx, 0)
                    Nx = fr.shape[1]
                    dx = torch.from_numpy(np.ascontiguousarray(fr)).to(dev_t)
                    with api.ConesGpu(max_points=Fx * Nx, max_frames=Fx, device=dev_index) as hx:
                        hx.set_device_input(dx.data_ptr(), np.full(Fx, Nx, np.uint32), keep=dx)
                        for _ in range(4):
                            hx.run(cfgx.detect, cfgx.ground)
                            hx.sync()
                        cx, ox, _ = hx.results()
                        lat_ = []
                        for _ in range(20):
                            t_ = time.perf_counter()
                            hx.run(cfgx.detect, cfgx.ground)
                            hx.sync()
                            lat_.append(1e3 * (time.perf_counter() - t_))
                        msx = float(np.percentile(lat_, 50))
                        Px = (int(cx["key_bits"].max()) + 7) // 8
                        Cx, Vx, Kx = int(cx["n_cropped"].sum()), int(cx["n_voxels"].sum()), int(cx["n_clusters"].sum())
                        b_alg = (32 if cfgx.ground is not None else 16) * Fx * Nx + (72 + 16 * Px) * Cx + 104 * Vx + 16 * Kx
                        rec["single" if Fx == 1 else "batch8"] = {
                            "ms_per_frame": msx / Fx, "points_per_frame": Nx, "C": Cx // Fx, "V": Vx // Fx, "K": Kx // Fx,
                            "launches": hx.last_launch_count(), "b_alg_bytes_per_frame": b_alg // Fx,
                            "GBps": b_alg / (msx * 1e-3) / 1e9, "frac_of_peak": b_alg / (msx * 1e-3) / 1e9 / peak}
                    del dx
                rec["what"] = ("dense 128-beam x 10-sweep cloud, fsai params" if idx == 4 else
                               "adversarial clustering (fences, 10.6k-voxel chain, solid blobs), simulation params") + \
                              "; p50 of 20 runs through cp_batch_run + cp_sync, device-resident"
                subs[f"cfg{idx}"] = rec

    line = None
    if rank == 0:
        # ---- single-frame latency (config 2): host cloud in -> cone list out
        cfg2 = scans.config(2)
        f2 = scans.generate(cfg2, 1, base_seed=0)[0]
        pin = torch.empty((N, 4), dtype=torch.float32, pin_memory=True)
        pin.numpy()[:] = f2
        lat_gpu = api.ConesGpu(max_points=N, max_frames=1, device=dev_index)
        m2 = PointCloud2.from_xyzi(pin.numpy())
        for _ in range(5):
            cl2, _ = lat_gpu.detect(m2, cfg2.detect, cfg2.ground)
        # timed through the C ABI itself (cp_detect) with the arguments prepared once, as the C++ node calls it;
        # the ctypes wrapper's per-call conversions (about 6 us) are the binding's, not the library's
        import ctypes as C
        from cones_perception_b200.params import to_c_detect, to_c_ground
        from cones_perception_b200.pointcloud2 import make_view
        view2 = make_view(m2, True)
        cd2, cg2 = to_c_detect(cfg2.detect), to_c_ground(cfg2.ground)
        out2 = np.zeros(4096, dtype=api.CLUSTER_DTYPE)
        ctr2 = np.zeros(1, dtype=api.COUNTER_DTYPE)
        k2 = C.c_uint32()
        cargs = (lat_gpu._h, C.byref(view2), C.byref(cd2), C.byref(cg2), out2.ctypes.data, 4096, C.byref(k2),
                 ctr2.ctypes.data)
        lat = []
        for _ in range(args.latency_reps):
            t = time.perf_counter()
            st = lat_gpu.lib.cp_detect(*cargs)
            lat.append(1e3 * (time.perf_counter() - t))
            assert st == 0
        assert k2.value == len(cl2) and np.array_equal(out2[:k2.value].view(np.uint32), cl2.view(np.uint32))
        lat_launches = lat_gpu.last_launch_count()
        # the same from pageable memory (a ROS message's std::vector): staged through the library's pinned ring
        m2p = PointCloud2.from_xyzi(f2.copy())
        lat_page = []
        for i in range(3 + args.latency_reps):
            t = time.perf_counter()
            lat_gpu.detect(m2p, cfg2.detect, cfg2.ground)
            if i >= 3:
                lat_page.append(1e3 * (time.perf_counter() - t))
        # the two-node configuration of the reference (cones_perception.launch, ground_removal:=true): the ground
        # node alone (cp_ground_remove: cloud in, N x 32 B PCL cloud out) and the detection node on that 32-byte
        # cloud without ground removal — what a drop-in of the two separate nodes pays per frame
        lat_ground, lat_det32 = [], []
        g_out = None
        for i in range(3 + args.latency_reps):
            t = time.perf_counter()
            g_out, _, _ = lat_gpu.ground_remove(m2, cfg2.ground, copy=False)
            if i >= 3:
                lat_ground.append(1e3 * (time.perf_counter() - t))
        from cones_perception_b200.pointcloud2 import PointField
        pin32 = torch.empty((N, 8), dtype=torch.float32, pin_memory=True)
        pin32.numpy()[:] = g_out
        m32 = PointCloud2(width=N, height=1, point_step=32, row_step=32 * N,
                          fields=[PointField("x", 0), PointField("y", 4), PointField("z", 8), PointField("intensity", 16)],
                          data=pin32.numpy().view(np.uint8).reshape(-1))
        lat32 = api.ConesGpu(max_points=N, max_frames=1, device=dev_index, max_point_step=32)
        for i in range(3 + args.latency_reps):
            t = time.perf_counter()
            cl32, _ = lat32.detect(m32, cfg2.detect, None)
            if i >= 3:
                lat_det32.append(1e3 * (time.perf_counter() - t))
        assert np.array_equal(cl32.view(np.uint32), cl2.view(np.uint32)), "chained nodes and fused detection disagree"
        lat32.close()
        d2 = torch.from_numpy(f2).cuda()
        lat_gpu.set_device_input(d2.data_ptr(), np.array([N], np.uint32), keep=d2)
        lat_dev = []
        for _ in range(args.latency_reps):
            t = time.perf_counter()
            lat_gpu.run(cfg2.detect, cfg2.ground)
            lat_gpu.sync()
            lat_dev.append(1e3 * (time.perf_counter() - t))
        lat_gpu.close()

        # ---- CPU baseline beside it (rank 0, N = 1 only): one core, bounded sample
        cpu = None
        if world == 1 and args.cpu_sample_frames > 0:
            ns = min(args.cpu_sample_frames, F)
            dt, stages, passes = 0.0, None, 0
            kept = [None] * ns
            while dt < args.cpu_sample_seconds and passes < 8:      # about 10 s of single-core work
                d1, stages = cpu_frames_per_sec(hnp[:ns], cfg, threads=1, keep=kept if passes == 0 else None)
                dt += d1
                passes += 1
            # parity of the TIMED batch: the oracle's clusters for these frames against the GPU step's results
            parity = compare_with_oracle(kept, ctr, k_off, clusters)
            # the ground node's two atan2f per point are most of the CPU time: the oracle's restated fdlibm routine
            # next to this box's libm on one frame's (y, x) pairs, so the baseline is seen not to be sandbagged
            from oracle import oracle as O
            yx = np.ascontiguousarray(hnp[0, :, 1]), np.ascontiguousarray(hnp[0, :, 0])
            t_or = min(O.time_atan2f(yx[0], yx[1], False) for _ in range(5))
            t_lm = min(O.time_atan2f(yx[0], yx[1], True) for _ in range(5))
            atan_note = {"restated_ns_per_call": 1e9 * t_or / N, "libm_ns_per_call": 1e9 * t_lm / N,
                         "calls_per_point": 2}
            cpu = {"value": passes * ns * N / dt, "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"first {ns} frames of the step's batch x {passes} passes, oracle pcl_faithful mode "
                             f"(PCL cost profile), g++ -O2, single thread like the reference's ros::spin nodes",
                   "frames_per_sec": passes * ns / dt, "ms_per_frame": 1e3 * dt / (passes * ns),
                   "stage_ms_per_frame": stages,
                   "host_cores_available": os.cpu_count(), "parity_of_timed_batch": parity,
                   "atan2f": atan_note, "host": host_description()}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "frames_per_sec": value / N,
            "p50_frame_latency_ms": float(np.percentile(lat, 50)), "p99_frame_latency_ms": float(np.percentile(lat, 99)),
            "p50_frame_latency_pageable_ms": float(np.percentile(lat_page, 50)),
            "p99_frame_latency_pageable_ms": float(np.percentile(lat_page, 99)),
            "p50_frame_latency_device_resident_ms": float(np.percentile(lat_dev, 50)),
            "p99_frame_latency_device_resident_ms": float(np.percentile(lat_dev, 99)),
            "latency_launches_per_frame": lat_launches,
            "two_node_configuration": {
                "p50_ground_node_ms": float(np.percentile(lat_ground, 50)),
                "p50_detection_node_on_32B_cloud_ms": float(np.percentile(lat_det32, 50)),
                "what": "cp_ground_remove (pinned cloud in, N x 32 B PCL cloud out) and cp_detect on that cloud "
                        "without ground removal, through the Python wrapper; the fused call above does both"},
            "config": {**workload_config(F, N, world),
                       "parallelism": f"frames sharded over {world} GPU(s), no data-path collective; when N>1 every "
                                      "rank publishes its cone list into rank 0's memory (CUDA-IPC peer stores over "
                                      "NVLink), NCCL for setup / barriers only",
                       "result_gather": gather_mode, "result_gather_check": gather_check,
                       "batches_in_flight": len(lanes),
                       "cache": f"inputs larger than L2 ({F * N * 16 / 1e6:.0f} MB per rank vs 126 MB), no flush needed",
                       "latency_workload": "cfg2 single frame, host cloud in -> cone list out"},
            "per_step_counts": {"points": F * N, "cropped": C_tot, "voxels": V_tot, "clusters": K_tot},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "sub_records": subs,
            "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
            "clocks": clocks,
        }
    for h in lanes:
        h.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if line is not None:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--frames-per-gpu", type=int, default=512)
    ap.add_argument("--latency-reps", type=int, default=200)
    ap.add_argument("--lanes", type=int, default=4, help="batches in flight (handles/streams alternating per step)")
    ap.add_argument("--cpu-sample-frames", type=int, default=512, help="frames timed on one core for cpu_baseline")
    ap.add_argument("--cpu-sample-seconds", type=float, default=10.0, help="minimum CPU time spent on cpu_baseline")
    ap.add_argument("--no-sub-records", dest="sub_records", action="store_false",
                    help="skip rowskip_off / azimuth_major / strong_4096 / cfg4 / cfg5")
    ap.add_argument("--strong-frames", type=int, default=4096, help="global batch of the strong-scaling sub-record")
    ap.add_argument("--cpu-step-frames", type=int, default=0,
                    help="frames per step of --impl reference (0 = --frames-per-gpu, the CUDA arm's batch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's counters, cluster offsets and clusters as "
                         "DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's results (--impl ours)")
    if args.dump_outputs and os.path.isdir(args.dump_outputs) and os.listdir(args.dump_outputs):
        # files of an earlier run (another --gpus, a sample) would sit beside the new ones and be compared too
        ap.error(f"--dump-outputs {args.dump_outputs} is not empty")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
