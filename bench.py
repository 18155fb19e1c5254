#!/usr/bin/env python
"""bench.py — rend3 hot path on B200: culled objects/s (cull + uniform bake) and shaded Mfrag/s (PBR forward).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU arithmetic (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed as DIR/<name>.npy

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch of synthetic input:
  * headline workload (BASELINE config 4, the one the target metric is quoted on): fused per-object frustum cull +
    object-uniform bake over 10 M object records PER GPU (weak scaling), 1% disabled, visible list ascending;
    at N > 1 every rank receives the visible set of all shards (1 bit per object) through peer-memory stores fused into the
    compaction kernel, published with per-row epoch flags (r3_exchange_*), and a consumer kernel chained on those flags counts
    every shard's visible objects — no host barrier, no collective kernel; `with_global_list` is the same step with the rows
    also expanded into the global visible list on every rank (an output that grows with the number of ranks);
  * `value` = objects culled+baked per second, inputs resident in HBM, CUDA events on the library's stream;
  * `strong_scaling` = BASELINE config 4 as stated: 10 M objects in TOTAL, 10 M / N per GPU;
  * `e2e`   = the same through the C ABI with HOST buffers: r3_set_objects (pinned H2D of every record) +
    r3_object_uniform_upload + r3_readback_visible (D2H) inside the timed region; `dynamic` = the sparse-update path
    (r3_update_objects of 1% / 10% / 100% of the records per step + cull + bake);
  * `forward` = BASELINE config 5 (4K, ~500k triangles, 64 point lights + 4 shadow-mapped directional lights):
    whole frames through BaseRenderGraph.add_to_graph; Mfrag/s = fs_main invocations / frame time; per-kernel rooflines from
    the library's stage timer; at N > 1 the screen is split in row tiles, one per rank.
Inputs (0.8 GB of transforms + spheres read, 1.28 GB of matrices written per step) exceed the 126 MB L2, so no explicit
flush is needed.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from rend3_b200.backend import CAMERA_VIEWPORT, CB_BAKE, CB_CULL  # noqa: E402
from rend3_b200.layouts import OBJECT_MATRICES_DTYPE  # noqa: E402
from rend3_b200.routines import BaseRenderGraph, BaseRenderGraphSettings, per_camera_header  # noqa: E402
from rend3_b200.scenes import cloud_camera, cube_field_scene, object_cloud_records  # noqa: E402

METRIC = "culled objects/s (fused frustum cull + object-uniform bake)"
BYTES_PER_OBJECT = 212   # SURVEY 8d: 84 B read (transform 64 + sphere 16 + enabled 4) + 128 B MV/MVP written
BYTES_PER_VISIBLE = 4
TRI_TEST_BYTES = 66      # SURVEY 8d: ~60-72 B per tested triangle (12 B indices + 36 B positions + MVP / batch entry share + bits)
SETUP_COLOUR_BYTES = 112  # per listed triangle: 12 B indices + 36 B positions + 64 B triangle record written
SETUP_DEPTH_BYTES = 48    # depth-only: 12 B indices + 36 B positions
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # 148 SMs x 128 FP32 lanes x 2 flop (FMA) x 1.965 GHz boost


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def kernel_source_sha():
    """Identity of the cull + bake kernel source: a DRAM-traffic capture only counts when it was taken from this source."""
    h = hashlib.sha256()
    for f in ("rend3_b200/csrc/r3_cull_bake.cu", "rend3_b200/csrc/r3_common.cuh"):
        h.update(open(os.path.join(ROOT, f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(n_objects):
    """dram__bytes_read.sum + dram__bytes_write.sum of cull_bake_kernel from the capture tools/capture_traffic.py wrote
    (profiles/ncu_cull_bake_traffic.json).  Returns (bytes per launch or None, provenance).  No literals: a capture taken from
    another kernel source (sha mismatch) or a missing file yields null."""
    p = os.path.join(ROOT, "profiles", "ncu_cull_bake_traffic.json")
    if not os.path.exists(p):
        return None, "no capture (run tools/capture_traffic.py under gpurun)"
    try:
        cap = json.load(open(p))
        if cap.get("kernel_source_sha16") != kernel_source_sha():
            return None, f"stale capture ({p}: taken from another kernel source)"
        per_object = (cap["dram_bytes_read"] + cap["dram_bytes_write"]) / cap["objects"]
        return per_object * n_objects, f"profiles/ncu_cull_bake_traffic.json ({cap['objects']} objects, ncu --set full, kernel source {cap['kernel_source_sha16']}), scaled per object"
    except Exception as e:   # noqa: BLE001
        return None, f"unreadable capture: {e}"


# --dump-outputs: at most 32 MB of visible list + 8 MB of matrices + 18 MB of frame samples, under 64 MB in all
DUMP_VISIBLE_BYTES = 32 << 20
DUMP_MATRIX_OBJECTS = 1 << 16
DUMP_PIXELS = 1 << 19


def seeded_sample(n, k, seed):
    """Ascending positions of a fixed sample of k out of n (all n when n <= k), the same on every run."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_cull_bake(out_dir, backend, enabled):
    """What a caller of the cull + bake step receives: the visible-object count, the ascending visible list (a fixed sample of its
    positions past DUMP_VISIBLE_BYTES) and MV / MVP of a fixed sample of the enabled objects (disabled slots hold no defined matrices)."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(enabled)
    vis = backend.readback_visible(CAMERA_VIEWPORT)
    id_type = np.float32 if n <= 1 << 24 else np.float64   # object ids stay exact
    np.save(os.path.join(out_dir, "visible_count.npy"), np.array([len(vis)], dtype=np.float64))
    np.save(os.path.join(out_dir, "visible_objects.npy"),
            vis[seeded_sample(len(vis), DUMP_VISIBLE_BYTES // np.dtype(id_type).itemsize, 1)].astype(id_type))
    ids = np.flatnonzero(enabled)
    ids = ids[seeded_sample(len(ids), DUMP_MATRIX_OBJECTS, 2)]
    chunk, parts = 1 << 20, []
    for first in range(0, n, chunk):      # chunked so that the host copies stay small
        sel = ids[(ids >= first) & (ids < first + chunk)]
        if len(sel):
            parts.append(backend.readback_object_matrices(CAMERA_VIEWPORT, first, int(sel[-1]) + 1 - first)[sel - first])
    mats = np.concatenate(parts) if parts else np.zeros(0, dtype=OBJECT_MATRICES_DTYPE)
    np.save(os.path.join(out_dir, "object_model_view.npy"), mats["model_view"].astype(np.float32))
    np.save(os.path.join(out_dir, "object_model_view_proj.npy"), mats["model_view_proj"].astype(np.float32))


def dump_frame(out_dir, backend):
    """What a caller of the forward path receives, at a fixed sample of pixels: the tonemapped target, the HDR colour and the depth."""
    os.makedirs(out_dir, exist_ok=True)
    px = seeded_sample(backend.width * backend.height, DUMP_PIXELS, 3)
    np.save(os.path.join(out_dir, "frame_ldr.npy"), backend.readback_ldr().reshape(-1, 4)[px].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_hdr.npy"), backend.readback_hdr_f16().reshape(-1, 4)[px].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_depth.npy"), backend.readback_depth().reshape(-1)[px].astype(np.float32))


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md's clocks line).  The timed region of this
    workload is a few milliseconds, far shorter than one `nvidia-smi` invocation, so the sampler polls NVML directly
    (nvidia_ml_py: the library nvidia-smi itself reads) every ~0.5 ms and only falls back to nvidia-smi without it."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, uuid=None):
        self.index, self.rows, self.stop, self.nvml, self.handle, self.source = index, [], False, None, None, "nvidia-smi"
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid if str(uuid).startswith("GPU-") else f"GPU-{uuid}") if uuid else None
            except Exception:
                self.handle = None
            if self.handle is None:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml"
        except Exception:
            self.nvml = None
        self.t = threading.Thread(target=self.run, daemon=True)

    def sample(self):
        if self.nvml is not None:
            n = self.nvml
            sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            try:
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.rows.append((sm, self.max_mhz, mask, time.perf_counter()))
            return
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            c = [x.strip() for x in out.split(",")]
            mask = sum(bit for k, bit in zip(range(2, 6), (0x8, 0x40, 0x20, 0x4)) if len(c) > k and c[k].lower().startswith("active"))
            self.rows.append((float(c[0]), float(c[1]), mask, time.perf_counter()))

    def run(self):
        while not self.stop:
            try:
                self.sample()
            except Exception:
                pass
            time.sleep(0.0002 if self.nvml is not None else 0.1)

    def sample_now(self):
        try:
            self.sample()
        except Exception:
            pass

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def summary(self):
        """Samples stamped inside [mark_begin, mark_end] (the timed region).  The region is only milliseconds long, so when
        fewer than 3 samples fell inside it the nearest samples of the surrounding warm-up / drain (same workload) are added."""
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0, "source": self.source}
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", float("inf"))
        inside = [r for r in self.rows if t0 <= r[3] <= t1]
        used = inside
        if len(inside) < 3:
            mid = 0.5 * (t0 + min(t1, self.rows[-1][3]))
            used = sorted(self.rows, key=lambda r: abs(r[3] - mid))[:max(3, len(inside))]
        sm = sorted(r[0] for r in used)
        mask = 0
        for r in used:
            mask |= r[2]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": used[0][1], "reasons": [k for k, bit in self.BITS.items() if mask & bit],
                "samples": len(used), "samples_in_timed_region": len(inside), "source": self.source}


class DeviceView:
    """__cuda_array_interface__ wrapper so torch.distributed can move library-owned device memory without a host bounce."""

    def __init__(self, ptr, nbytes, typestr="|u1", itemsize=1):
        self.__cuda_array_interface__ = {"shape": (nbytes // itemsize,), "typestr": typestr, "data": (ptr, False), "version": 2}


# ---------------------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def best_thread_count(oracle, backend, header, n_sample):
    """The oracle's OpenMP loop is memory-bound: more threads than memory channels (or than a cgroup quota grants) make it slower.
    A short sweep on a sample picks the count the timed run then uses ("all the host threads it can use")."""
    best, best_rate, tried = 1, 0.0, {}
    hw = host_threads()
    for t in sorted({1, 4, 8, 16, 32, 64, hw}):
        if t > hw:
            continue
        oracle.set_threads(t)
        backend.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
        dt = float("inf")
        for _ in range(3):           # best of three: a single call is at the mercy of whatever else the host is doing
            t0 = time.perf_counter()
            backend.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
            dt = min(dt, time.perf_counter() - t0)
        rate = n_sample / dt
        tried[t] = rate
        if rate > best_rate:
            best, best_rate = t, rate
    oracle.set_threads(best)
    return best, tried


def single_thread_batch_objects(n):
    """SURVEY 8d: the reference's real object-level path — batch_objects (frustum filter, sort, batch build) — is single-threaded under
    the data_core mutex (batching.rs:120-250 below graph.rs:265).  Timed here on ONE host thread over the same object set."""
    import oracle

    oracle.set_threads(1)
    rec = object_cloud_records(n, seed=4)
    header = per_camera_header(cloud_camera(), CAMERA_VIEWPORT, (1920, 1080), 1, n)
    b = oracle.load_oracle_backend()
    b.set_objects(rec)
    b.set_object_sort_info(np.zeros(n, dtype=np.uint64), np.full(n, 3, dtype=np.uint8), rec["sphere_center"])
    t0 = time.perf_counter()
    b.object_uniform_upload(CAMERA_VIEWPORT, header, CB_CULL)            # the sphere-frustum filter of batching.rs:144-148
    t1 = time.perf_counter()
    b.batch_objects(CAMERA_VIEWPORT, np.zeros(3, dtype=np.float32))      # sort_unstable_by_key + batch build (batching.rs:175-247)
    t2 = time.perf_counter()
    nb, nr, _ = b.batch_counts(CAMERA_VIEWPORT)
    return {"objects": n, "visible": int(b.visible_count(CAMERA_VIEWPORT)), "filter_s": t1 - t0, "sort_and_batch_s": t2 - t1,
            "objects_per_s": n / (t2 - t0), "batches": nb, "regions": nr, "threads": 1,
            "what": "oracle restatement of batch_objects on one host thread: frustum filter + sort + ShaderBatchData build"}


def reference_arm(args):
    """The reference's own CPU arithmetic for the path.  The reference (Rust + wgpu) cannot be built or run here (no
    cargo, no Vulkan ICD: SURVEY 8c), so this arm times the oracle port — uniform_prep.wgsl + batch_objects' frustum filter
    restated in C — on the host cores, every step over the FULL per-GPU workload of our arm (same config)."""
    import oracle

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.objects
    rec = object_cloud_records(n, seed=4)
    header = per_camera_header(cloud_camera(), CAMERA_VIEWPORT, (1920, 1080), 1, n)
    b = oracle.load_oracle_backend()
    b.set_objects(rec)
    cores, sweep = best_thread_count(oracle, b, header, n)
    for _ in range(args.warmup):
        b.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        b.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_cull_bake(args.dump_outputs, b, rec["enabled"])
    value = n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "objects/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE config 4: fused frustum cull + uniform bake, 10 M object records per GPU (128 B std430 records, 1% disabled)",
                   "objects_per_gpu": n, "visible_fraction": b.visible_count(CAMERA_VIEWPORT) / n,
                   "note": "reference itself (Rust/wgpu) cannot run here; CPU oracle port of uniform_prep.wgsl + Frustum::contains_sphere, whole workload per step"},
        "cpu_baseline": {"value": value, "unit": "objects/s", "cores": cores, "kind": "port",
                         "sample": f"all {n} records per step, OpenMP threads picked by a sweep ({ {k: round(v / 1e6, 1) for k, v in sweep.items()} } M objects/s), host has {host_threads()} hardware threads"},
        "e2e": {"value": value, "unit": "objects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline(n_total):
    import oracle

    n = min(n_total, 4_000_000)
    rec = object_cloud_records(n, seed=4)
    header = per_camera_header(cloud_camera(), CAMERA_VIEWPORT, (1920, 1080), 1, n)
    b = oracle.load_oracle_backend()
    b.set_objects(rec)
    cores, sweep = best_thread_count(oracle, b, header, n)
    reps, t0 = 0, time.perf_counter()
    while reps < 3 or (time.perf_counter() - t0 < 4.0 and reps < 50):
        b.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    out = {"value": n / dt, "unit": "objects/s", "cores": cores, "kind": "port",
           "sample": f"{n} of {n_total} records, {reps} repetitions, OpenMP threads picked by a sweep over {sorted(sweep)} of {host_threads()} hardware threads (oracle/r3_oracle.c)"}
    del b, rec
    try:
        out["batch_objects_single_thread"] = single_thread_batch_objects(min(n_total, 2_000_000))
    except Exception as e:   # noqa: BLE001
        out["batch_objects_single_thread"] = {"error": str(e)}
    return out


# ---------------------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--objects", type=int, default=10_000_000, help="object records per GPU")
    ap.add_argument("--no-forward", action="store_true")
    ap.add_argument("--no-dynamic", action="store_true")
    ap.add_argument("--forward-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return reference_arm(args)
    # keep stdout clean for the single JSON line: anything libraries print (e.g. NCCL's version banner) goes to stderr
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    from rend3_b200 import load_cuda_backend   # fails loudly when librend3_b200.so is missing: no CPU fallback

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.objects
    backend = load_cuda_backend(local)
    stream = torch.cuda.ExternalStream(backend.stream(), device=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs: this rank's shard of the object set, built on the host, staged in pinned memory
    rec = object_cloud_records(n, seed=4 + rank)
    pinned = torch.empty(n * 128, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = rec.view(np.uint8).reshape(-1)
    host_rec = pinned.numpy().view(rec.dtype)
    del rec
    header = per_camera_header(cloud_camera(), CAMERA_VIEWPORT, (1920, 1080), 1, n)
    backend.set_objects(host_rec)
    vis_host = torch.empty(n, dtype=torch.int32, pin_memory=True)

    # ---- north-star exchange (N > 1): r3_exchange_* — the compaction kernel stores every visibility word into all ranks' buffers over
    # NVLink and publishes the row with an epoch flag (st.release.sys); r3_exchange_merge, a consumer kernel chained on the flags with
    # ld.acquire.sys, turns the rows into the GLOBAL visible list on every rank.  No host barrier between the steps.
    exchange, exchange_kind = None, "single GPU"
    if world > 1:
        from rend3_b200.parallel import VisibilityExchange
        try:
            exchange = VisibilityExchange(backend, CAMERA_VIEWPORT, n, rank, world)
            exchange_kind = "peer-memory stores fused into the compaction kernel + per-row epoch flags + a consumer kernel chained on the flags that counts every shard's visible objects (NVLink P2P, CUDA IPC)"
        except Exception as e:   # noqa: BLE001
            print(f"[rank {rank}] peer-memory exchange unavailable ({e})", file=sys.stderr)
            exchange = None
        ok = torch.tensor([1 if exchange is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            if exchange is not None:
                exchange.close()
            exchange, exchange_kind = None, "NCCL all-gather of the visibility words (peer-memory exchange unavailable on this box)"
    gathered_words = torch.empty(world * ((n + 31) // 32), dtype=torch.int32, device=dev) if world > 1 and exchange is None else None

    def step_resident(full_list=False):
        backend.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
        if world == 1:
            return
        if exchange is not None:
            # consumer kernels chained on the peers' epoch flags ON THE DEVICE: the headline step counts the visible objects of every shard
            # (it has to see every row of this epoch); `with_global_list` also expands the rows into the global visible list, whose size —
            # 4 B per visible object of the WHOLE world on every rank — grows with the number of ranks
            if full_list:
                exchange.merge()
            else:
                exchange.count()
        else:
            wptr, wbytes = backend.device_ptr(CAMERA_VIEWPORT, 4)
            with torch.cuda.stream(stream):
                mine = torch.as_tensor(DeviceView(wptr, wbytes, "<i4", 4), device=dev)
                dist.all_gather_into_tensor(gathered_words, mine)

    clocks = ClockSampler(local, getattr(torch.cuda.get_device_properties(local), "uuid", None))
    clocks.__enter__()               # polls through warm-up, timed region and drain; only the stamped window is reported
    for _ in range(args.warmup):
        step_resident()
    barrier()
    exchange_verified = None
    if exchange is not None:
        # outside the timed region: the merged global list must equal the one built from an NCCL all-gather of the same words, and the
        # light consumer's per-shard counts must add up to its length
        step_resident(full_list=True)
        exchange_verified = exchange.verify_against_nccl(stream, dev)
        n_list = int(exchange.merged(dev).numel())
        step_resident()
        counts = exchange.counts()
        exchange_verified = bool(exchange_verified and int(counts[-1]) == n_list and int(counts[:-1].sum()) == n_list)
        barrier()
    launches0 = backend.launch_count()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    clocks.mark_begin()
    for i in range(args.steps):
        starts[i].record(stream)
        step_resident()
        ends[i].record(stream)
    if exchange is not None:
        exchange.join()              # the consumer kernels run on the library's side stream: the main stream waits for the last ones here
    final = torch.cuda.Event(enable_timing=True)
    final.record(stream)
    clocks.sample_now()              # GPU busy with the queued steps
    barrier()
    clocks.mark_end()
    clocks.__exit__()
    # device time of the K steps on this rank (first start -> everything of the last step done); the job's time is the max over ranks
    total_ms = max_over_ranks(starts[0].elapsed_time(final))
    launches = backend.launch_count() - launches0
    n_vis = backend.visible_count(CAMERA_VIEWPORT)
    if args.dump_outputs and rank == 0:
        dump_cull_bake(args.dump_outputs, backend, host_rec["enabled"])
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3)
    peak, peak_src = measured_peak_gbs()

    # dominant kernel alone: the library's stage timer (CUDA events around cull_bake_kernel on its own stream), separate short pass
    backend.set_stage_timing(True)
    for _ in range(max(5, min(args.steps, 10))):
        backend.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
    st = backend.stage_times()["cull_bake"]
    backend.set_stage_timing(False)
    kern_s = st["ms"] / max(st["launches"], 1) * 1e-3
    algorithmic = BYTES_PER_OBJECT * n + BYTES_PER_VISIBLE * n_vis
    achieved = algorithmic / kern_s / 1e9
    traffic, traffic_src = measured_traffic(n)
    barrier()

    # ---- the same step with the global visible list expanded on every rank (r3_exchange_merge)
    with_list = None
    if exchange is not None:
        for _ in range(args.warmup):
            step_resident(full_list=True)
        barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        for _ in range(args.steps):
            step_resident(full_list=True)
        exchange.join()
        w1.record(stream)
        barrier()
        wms = max_over_ranks(w0.elapsed_time(w1)) / args.steps
        with_list = {"what": "cull + bake + exchange + the global ascending visible list built on every rank each step (4 B x visible objects of all shards)",
                     "ms_per_step": wms, "value": world * n / (wms * 1e-3), "unit": "objects/s", "list_entries": n_list, "list_bytes_per_rank_per_step": 4 * n_list}
        barrier()

    # ---- strong scaling: BASELINE config 4 as stated — 10 M objects in total, 10 M / N per GPU
    strong = None
    if world > 1:
        ns = n // world
        sheader = per_camera_header(cloud_camera(), CAMERA_VIEWPORT, (1920, 1080), 1, ns)

        def step_strong():
            backend.object_uniform_upload(CAMERA_VIEWPORT, sheader, CB_BAKE | CB_CULL)   # the first 10 M / N records of this rank's buffer
            if exchange is not None:
                exchange.count([ns] * world)
        for _ in range(args.warmup):
            step_strong()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(args.steps):
            step_strong()
        if exchange is not None:
            exchange.join()
        s1.record(stream)
        barrier()
        sms = max_over_ranks(s0.elapsed_time(s1)) / args.steps
        strong = {"workload": f"BASELINE config 4 as stated: {ns * world} objects in total, {ns} per GPU, visible set exchanged + counted on every rank",
                  "objects_total": ns * world, "ms_per_step": sms, "value": ns * world / (sms * 1e-3), "unit": "objects/s", "scaling": "strong"}
        for _ in range(2):   # back to the full shard (the exchange rows carry the 10 M-object words again)
            step_resident()
        barrier()

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region
    e2e_steps = max(3, min(args.steps, 5))
    backend.set_objects(host_rec)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        backend.set_objects(host_rec)                                         # pinned H2D of every record
        backend.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
        nv = backend.visible_count(CAMERA_VIEWPORT)
        backend._call("readback_visible", ctypes.c_uint32(CAMERA_VIEWPORT), ctypes.c_void_p(vis_host.data_ptr()), ctypes.c_uint32(n), None)   # D2H into pinned memory
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e = {"value": world * n / e2e_s, "unit": "objects/s", "h2d_bytes_per_step": n * 128 + 240, "d2h_bytes_per_step": 4 * nv + 4,
           "what": "worst case: every record re-uploaded each step (r3_set_objects), PCIe-bound"}

    # ---- dynamic: the realistic per-frame path — a fraction of the objects changes, r3_update_objects scatters them (ScatterCopy) and
    # refreshes their hot copies (split_slots_kernel), then cull + bake; H2D of the changed records + D2H of the count inside the timed region
    dynamic = None
    if not args.no_dynamic:
        dynamic = []
        rng = np.random.default_rng(11 + rank)
        for frac in (0.01, 0.1, 1.0):
            m = max(1, int(n * frac))
            slots_np = np.sort(rng.choice(n, m, replace=False)).astype(np.uint32) if frac < 1.0 else np.arange(n, dtype=np.uint32)
            slots = torch.empty(m, dtype=torch.int32, pin_memory=True)
            slots.numpy()[:] = slots_np.view(np.int32)
            recs = torch.empty(m * 128, dtype=torch.uint8, pin_memory=True)
            recs.numpy()[:] = host_rec[slots_np].view(np.uint8).reshape(-1)   # same values: the visible set stays comparable
            d_steps = 3 if frac >= 1.0 else max(3, min(args.steps, 8))

            def dyn_step():
                backend._call("update_objects", ctypes.c_void_p(slots.data_ptr()), ctypes.c_void_p(recs.data_ptr()), ctypes.c_uint32(m))
                backend.object_uniform_upload(CAMERA_VIEWPORT, header, CB_BAKE | CB_CULL)
                return backend.visible_count(CAMERA_VIEWPORT)
            dyn_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(d_steps):
                dyn_step()
            barrier()
            ds = max_over_ranks((time.perf_counter() - t0) / d_steps)
            dynamic.append({"updated_fraction": frac, "updated_objects_per_step": m, "ms_per_step": ds * 1e3, "value": world * n / ds, "unit": "objects/s",
                            "h2d_bytes_per_step": m * 132 + 240, "d2h_bytes_per_step": 4})
            del slots, recs

    # ---- forward: BASELINE config 5
    forward = None
    if not args.no_forward:
        try:
            forward = forward_section(args, torch, dist, load_cuda_backend, rank, world, local, dev, barrier, max_over_ranks)
        except Exception as e:   # noqa: BLE001 — the headline line must survive a failure of the secondary workload
            if world > 1:
                raise            # ranks must fail together: a half-finished collective would hang the others
            forward = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "objects/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE config 4: fused frustum cull + uniform bake, 10 M object records per GPU (128 B std430 records, 1% disabled)",
                       "objects_per_gpu": n, "visible_fraction": n_vis / n,
                       "parallelism": f"object-range shards x{world}; visible set (1 bit/object) exchanged by {exchange_kind}" if world > 1 else "single GPU",
                       "exchange_verified_against_nccl": exchange_verified,
                       "l2": "inputs (0.8 GB) + outputs (1.28 GB) per step exceed the 126 MB L2; no explicit flush"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src, "kernel": "cull_bake_kernel<bake,cull>", "kernel_ms": kern_s * 1e3,
                         "kernel_timing": f"library stage timer: CUDA events around the kernel on its own stream, mean of {st['launches']} launches",
                         "frac_by_traffic": (traffic / kern_s / 1e9 / peak) if traffic else None,
                         "note": "achieved uses ALGORITHMIC bytes (SURVEY 8d counts `enabled` as 4 B per object; it travels as 1 bit, so DRAM traffic is ~6% lower): frac can exceed 1.0 by that margin, frac_by_traffic is the DRAM-side fraction",
                         "algorithmic_bytes_per_launch": algorithmic, "step_frac": algorithmic / (ms_per_step * 1e-3) / 1e9 / peak if world == 1 else None,
                         "peak_source": peak_src},
            "cpu_baseline": cpu_baseline(n),
            "e2e": e2e, "dynamic": dynamic, "strong_scaling": strong, "with_global_list": with_list, "gpu_launches": launches, "clocks": clocks.summary(), "forward": forward,
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if exchange is not None:
        exchange.close()
    if world > 1:
        dist.destroy_process_group()


def camera_triangles(backend, ev, camera):
    """Triangles the per-triangle cull of `camera` really tests: sum of index_count / 3 over its visible objects."""
    vis = backend.readback_visible(camera)
    return int((ev.object_buffer["index_count"][vis] // 3).sum()) if len(vis) else 0


def forward_section(args, torch, dist, load_cuda_backend, rank, world, local, dev, barrier, max_over_ranks):
    res = (3840, 2160)
    ev = cube_field_scene(n_objects=4400, seed=5, resolution=res, extent=30.0, pull_back=7.0, n_point_lights=64, n_dir_lights=4,
                          shadow_resolution=2048, shadow_distance=200.0, subdivisions=(2, 3, 3, 4), scale_range=(0.6, 2.4), slabs=True)
    fb = load_cuda_backend(local)
    fstream = torch.cuda.ExternalStream(fb.stream(), device=torch.device("cuda", local))
    graph = BaseRenderGraph(fb)
    settings = BaseRenderGraphSettings(clear_color=(0.1, 0.05, 0.1, 1.0))
    rows = (res[1] * rank // world, res[1] * (rank + 1) // world)
    n_shadows = len(ev.shadows)
    split = None
    if world > 1:
        from rend3_b200.parallel import ForwardSplit
        # the viewport's triangle test is 2% of this frame (config 5: 50 us): sharding it across the ranks (r3_set_cull_shard; exercised by
        # tests/test_multi_gpu.py) would add a flag round trip per frame for nothing — it pays on config-3-like scenes, so it stays off here
        split = ForwardSplit(fb, fstream, dev, rank, world, res, n_shadows, shard_triangle_cull=False)
        split.bind_scene(ev)

    def frame(upload):
        if world > 1:
            graph.add_to_graph(ev, res, 1, settings, upload=upload, scissor_rows=rows, shadow_filter=split.owns_shadow,
                               after_shadows=split.send_shadow_maps if n_shadows else None, before_resolve=split.wait_shadow_maps if n_shadows else None,
                               after_target=split.begin_frame, tonemap=False)
            split.exchange_rows(rows)
        else:
            # one GPU: the frame is recorded and submitted as ONE CUDA graph launch (r3_frame_begin / r3_frame_end), like the reference's
            # single queue submission per frame (graph.rs:510)
            graph.add_to_graph(ev, res, 1, settings, upload=upload, frame_graph=True)

    split_verified = None
    if world > 1 and res[1] % world == 0:
        # outside the timed region: the frame assembled from the ranks' row tiles and exchanged shadow maps must equal, bit for bit,
        # the frame one GPU renders alone
        frame(True)
        barrier()
        ptr, nbytes = fb.device_ptr(CAMERA_VIEWPORT, 1)
        got = torch.as_tensor(DeviceView(ptr, nbytes), device=dev).clone()
        vb = load_cuda_backend(local)
        BaseRenderGraph(vb).add_to_graph(ev, res, 1, settings)
        vb.sync()
        vptr, vbytes = vb.device_ptr(CAMERA_VIEWPORT, 1)
        want = torch.as_tensor(DeviceView(vptr, vbytes), device=dev)
        ok = torch.equal(got, want) if split.assembles_on(rank) else True
        same = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        split_verified = bool(int(same.item()))
        vb.close()
    frame(True)
    for _ in range(2):
        frame(False)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = fb.launch_count()
    f0.record(fstream)
    for _ in range(args.forward_steps):
        frame(False)
    f1.record(fstream)
    barrier()
    frame_ms = max_over_ranks(f0.elapsed_time(f1) / args.forward_steps)
    if args.dump_outputs and world == 1:   # with several ranks each one holds only its own rows of the frame
        dump_frame(args.dump_outputs, fb)
    launches_per_frame = (fb.launch_count() - l0) // max(args.forward_steps, 1)
    st = torch.tensor([float(x) for x in fb.forward_stats()[:3]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(st, op=dist.ReduceOp.SUM)
    tris = int(fb.readback_draw_calls(CAMERA_VIEWPORT, 0)["vertex_count"].sum()) // 3
    batching = fb.batching_info(CAMERA_VIEWPORT)

    # per-kernel rooflines of one GPU's frame (rank 0 reports its own kernels): durations from the library's stage timer
    fb.set_stage_timing(True)
    t_frames = 3
    for _ in range(t_frames):
        frame(False)
    times = fb.stage_times()
    fb.set_stage_timing(False)
    barrier()
    light_evals = fb.forward_light_evaluations()
    shaded_local = fb.forward_stats()[2]
    cams = [CAMERA_VIEWPORT] + [i for i in range(n_shadows) if split is None or split.owns_shadow(i)]
    tested = sum(camera_triangles(fb, ev, cam) for cam in cams)
    listed_colour = sum(int(fb.readback_draw_calls(CAMERA_VIEWPORT, part)["vertex_count"].sum()) // 3 for part in (0, 1))
    listed_depth = sum(int(fb.readback_draw_calls(i, 0)["vertex_count"].sum()) // 3 for i in cams[1:])
    peak, _ = measured_peak_gbs()

    def per_frame(stage):
        return times[stage]["ms"] / t_frames

    def hbm_block(stage, units, bytes_per_unit, what):
        ms = per_frame(stage)
        ach = units * bytes_per_unit / (ms * 1e-3) / 1e9 if ms > 0 else None
        return {"bound": "hbm (algorithmic bytes; the working set is L2-resident, so the kernel is issue-bound in practice)", "kernel_ms_per_frame": ms,
                "launches_per_frame": times[stage]["launches"] // t_frames, "units": units, "unit_name": what, "algorithmic_bytes_per_unit": bytes_per_unit,
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if ach else None}
    n_dir = n_shadows
    flops = shaded_local * 60.0 + light_evals * 95.0 + shaded_local * n_dir * 45.0   # SURVEY 8d: 60 + 95 per evaluated light + 45 per PCF5 shadow sample
    r_ms = per_frame("resolve")
    rooflines = {
        "triangle_test_kernel": hbm_block("triangle_test", tested, TRI_TEST_BYTES, "triangles tested (all cameras of this rank)"),
        "raster_setup_kernel<colour>": hbm_block("raster_setup_colour", listed_colour, SETUP_COLOUR_BYTES, "listed triangles (predicted + residual)"),
        "raster_setup_kernel<depth>": hbm_block("raster_setup_depth", listed_depth, SETUP_DEPTH_BYTES, "listed triangles (shadow passes of this rank)"),
        "resolve_kernel": {"bound": "fp32", "kernel_ms_per_frame": r_ms, "fragments": int(shaded_local), "light_evaluations": int(light_evals),
                           "lights_evaluated_per_fragment": light_evals / max(shaded_local, 1), "flop_model": "60 + 95 per evaluated light + 45 per shadowed directional light (SURVEY 8d)",
                           "achieved": flops / (r_ms * 1e-3) / 1e12 if r_ms > 0 else None, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s",
                           "frac": flops / (r_ms * 1e-3) / 1e12 / FP32_PEAK_TFLOPS if r_ms > 0 else None,
                           "peak_source": "148 SMs x 128 lanes x 2 x 1.965 GHz (nominal FP32 FMA rate)", "bytes_per_pixel": "8 B key read + 12 B written (rgba16f + depth32f)"},
        "other_stage_ms_per_frame": {k: per_frame(k) for k in ("raster_bands", "sort", "cull_bake", "triangle_compact")},
    }
    out = {"workload": "BASELINE config 5: 3840x2160, 4400 meshes / ~500k triangles, 64 point lights + 4 directional lights with 2048^2 shadow maps",
           "frame_ms": frame_ms, "shaded_mfrag_s": float(st[2].item()) / frame_ms / 1e3, "raster_mfrag_s": float(st[1].item()) / frame_ms / 1e3,
           "shaded_fragments": int(st[2].item()), "depth_passing_fragments": int(st[1].item()), "triangles_after_cull": tris,
           "gpu_launches_per_frame": launches_per_frame, "submission": (fb.frame_graph_stats() if world == 1 else "call by call (multi-GPU split)"), "batch_objects": batching,
           "split": split.describe() if split is not None else "single GPU", "split_equals_single_gpu_frame": split_verified,
           "timing": "CUDA events on the library stream around the timed frames, max over ranks", "roofline": rooflines}
    if split is not None:
        split.close()
    # BASELINE config 3 (single GPU only): the bistro-shaped scene — where the triangle cull and the shadow set-up dominate
    if world == 1:
        try:
            out["config3"] = config3_block(args, torch, load_cuda_backend, local)
        except Exception as e:   # noqa: BLE001
            out["config3"] = {"error": str(e)}
    return out


def config3_block(args, torch, load_cuda_backend, local):
    from rend3_b200 import configs

    ev, res = configs.config3()
    b = load_cuda_backend(local)
    s = torch.cuda.ExternalStream(b.stream(), device=torch.device("cuda", local))
    g = BaseRenderGraph(b)
    settings = BaseRenderGraphSettings(clear_color=(0.1, 0.05, 0.1, 1.0))
    g.add_to_graph(ev, res, 1, settings, upload=True, frame_graph=True)
    for _ in range(3):
        g.add_to_graph(ev, res, 1, settings, upload=False, frame_graph=True)
    b.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = b.launch_count()
    e0.record(s)
    for _ in range(args.forward_steps):
        g.add_to_graph(ev, res, 1, settings, upload=False, frame_graph=True)
    e1.record(s)
    b.sync()
    ms = e0.elapsed_time(e1) / args.forward_steps
    st = b.forward_stats()
    launches = (b.launch_count() - l0) // max(args.forward_steps, 1)
    b.set_stage_timing(True)
    for _ in range(2):
        g.add_to_graph(ev, res, 1, settings, upload=False)
    times = b.stage_times()
    b.set_stage_timing(False)
    cams = [CAMERA_VIEWPORT] + list(range(len(ev.shadows)))
    tested = sum(camera_triangles(b, ev, cam) for cam in cams)
    peak, _ = measured_peak_gbs()
    tt_ms = times["triangle_test"]["ms"] / 2
    out = {"workload": "BASELINE config 3: 200k objects over 1000 meshes (~20 M triangles), 4 shadow maps 2048^2 + 4 point lights, 3840x2160",
           "frame_ms": ms, "shaded_mfrag_s": st[2] / ms / 1e3, "shaded_fragments": int(st[2]), "gpu_launches_per_frame": launches, "batch_objects": b.batching_info(CAMERA_VIEWPORT),
           "stage_ms_per_frame": {k: v["ms"] / 2 for k, v in times.items()},
           "triangle_test_roofline": {"triangles_tested": tested, "algorithmic_bytes_per_triangle": TRI_TEST_BYTES, "kernel_ms_per_frame": tt_ms,
                                      "achieved": tested * TRI_TEST_BYTES / (tt_ms * 1e-3) / 1e9 if tt_ms > 0 else None, "peak": peak, "unit": "GB/s",
                                      "frac": tested * TRI_TEST_BYTES / (tt_ms * 1e-3) / 1e9 / peak if tt_ms > 0 else None}}
    b.close()
    return out


if __name__ == "__main__":
    main()
