"""Time r3_generate_mipmaps on the GPU and the CPU oracle on the same work; prints one JSON line and writes it to
profiles/r3_mipmaps_bench.json (or --out).

Workloads, each larger than the B200's 126 MB L2 so that level 0 comes from HBM on every call:
  a) 64 x 2048^2 Rgba8UnormSrgb            (a glTF scene's colour maps)
  b) 256 glTF-like sizes in mixed formats  (odd sizes included: 1000x750, 1366x768, 2049x1025, 4097x3)
  c) 16 x 4096^2 Rgba16Float               (HDR maps)
Level 0 never changes between calls, so every call repeats exactly the same work.  Algorithmic bytes = level 0 read once + every
generated level written once.  Times: CUDA events over >= 20 calls after warm-up; the oracle is timed once per workload.
--profile FILE: afterwards, in a pass of its own, torch.profiler's CUDA kernel table of 5 calls per workload is written to FILE."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rend3_b200 import layouts as L  # noqa: E402
from rend3_b200.backend import load_cuda_backend  # noqa: E402

BPP = {L.TEXFMT_RGBA8_UNORM: 4, L.TEXFMT_RGBA8_UNORM_SRGB: 4, L.TEXFMT_BGRA8_UNORM_SRGB: 4, L.TEXFMT_R8_UNORM: 1, L.TEXFMT_RG8_UNORM: 2,
       L.TEXFMT_RGB10A2_UNORM: 4, L.TEXFMT_RG16_FLOAT: 4, L.TEXFMT_RGBA16_FLOAT: 8}
DATASHEET_HBM_GBS = 7700.0


def table(specs, seed):
    descs = np.zeros(len(specs), dtype=L.TEXTURE_DESC_DTYPE)
    cursor, level0, generated = 0, 0, 0
    offsets = []
    for i, (fmt, w, h) in enumerate(specs):
        mips = max(w, h).bit_length()
        sizes = [max(w >> l, 1) * max(h >> l, 1) * BPP[fmt] for l in range(mips)]
        descs[i]["width"], descs[i]["height"], descs[i]["mip_count"], descs[i]["format"], descs[i]["byte_offset"] = w, h, mips, fmt, cursor
        offsets.append((cursor, sizes[0]))
        level0 += sizes[0]
        generated += sum(sizes[1:])
        cursor += sum(sizes) + (-sum(sizes)) % 16
    blob = np.zeros(cursor, dtype=np.uint8)
    rng = np.random.default_rng(seed)
    for o, n in offsets:
        blob[o: o + n] = rng.integers(0, 256, n, dtype=np.uint8)
    return descs, blob, level0, generated


def workloads():
    rng = np.random.default_rng(1)
    sizes = [(1000, 750), (1366, 768), (2049, 1025), (4097, 3), (2048, 2048), (1024, 1024), (512, 512), (1920, 1080), (800, 600), (300, 200), (4096, 2048), (1023, 1023)]
    fmts = list(BPP)
    mixed = [(fmts[rng.integers(len(fmts))],) + sizes[k % len(sizes)] for k in range(256)]
    return {
        "a_64x2048sq_rgba8_srgb": [(L.TEXFMT_RGBA8_UNORM_SRGB, 2048, 2048)] * 64,
        "b_256_gltf_mixed": mixed,
        "c_16x4096sq_rgba16f": [(L.TEXFMT_RGBA16_FLOAT, 4096, 4096)] * 16,
    }


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:   # noqa: BLE001 - reported, not fatal
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--oracle-threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_mipmaps_bench.json"))
    ap.add_argument("--profile", default=None, help="write torch.profiler kernel times of 5 calls per workload to this file")
    args = ap.parse_args()
    import torch

    import oracle
    import oracle_mipmaps

    threads = oracle.set_threads(args.oracle_threads)
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks):
        peak, peak_src = float(json.load(open(peaks))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = DATASHEET_HBM_GBS, "data-sheet HBM3e bandwidth (7.7 TB/s), not measured"
    line = {"tool": "bench_mipmaps", "gpu": card(), "peak_gbs": peak, "peak_source": peak_src, "calls": args.calls, "oracle_threads": threads, "workloads": {}}
    cuda = load_cuda_backend(0)
    stream = torch.cuda.ExternalStream(cuda.stream())
    for name, specs in workloads().items():
        descs, blob, level0, generated = table(specs, seed=len(specs))
        idx = np.arange(len(specs), dtype=np.uint32)
        cuda.set_textures(descs, blob)
        for _ in range(args.warmup):
            cuda.generate_mipmaps(idx)
        cuda.sync()
        n0 = cuda.launch_count()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for _ in range(args.calls):
            cuda.generate_mipmaps(idx)
        stop.record(stream)
        cuda.sync()
        ms = start.elapsed_time(stop) / args.calls
        launches = (cuda.launch_count() - n0) / args.calls
        gpu_out = cuda.readback_texels(0, len(blob))
        orc = oracle_mipmaps.load_oracle_backend()
        orc.set_textures(descs, blob)
        t0 = time.perf_counter()
        orc.generate_mipmaps(idx)
        oracle_ms = (time.perf_counter() - t0) * 1e3
        same = bool(np.array_equal(gpu_out, orc.readback_texels(0, len(blob))))
        orc.close()
        nbytes = level0 + generated
        gbs = nbytes / (ms * 1e-3) / 1e9
        line["workloads"][name] = {"textures": len(specs), "ms_per_call": round(ms, 4), "algorithmic_bytes": nbytes, "level0_bytes": level0,
                                   "generated_bytes": generated, "gbs": round(gbs, 1), "fraction_of_peak": round(gbs / peak, 3),
                                   "launches_per_call": launches, "oracle_ms": round(oracle_ms, 1), "bit_identical_to_oracle": same}
        del blob, gpu_out
    cuda.close()
    text = json.dumps(line)
    print(text)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    if args.profile:
        profile_kernels(args.profile, line["gpu"])


def profile_kernels(path, gpu):
    from torch.profiler import ProfilerActivity, profile

    cuda = load_cuda_backend(0)
    with open(path, "w") as f:
        f.write(f"# torch.profiler CUDA kernel times of r3_generate_mipmaps, 5 calls per workload (tools/bench_mipmaps.py --profile; {gpu})\n")
        for name, specs in workloads().items():
            descs, blob, level0, generated = table(specs, seed=len(specs))
            idx = np.arange(len(specs), dtype=np.uint32)
            cuda.set_textures(descs, blob)
            cuda.generate_mipmaps(idx)
            cuda.sync()
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(5):
                    cuda.generate_mipmaps(idx)
                cuda.sync()
            f.write(f"== {name}: {level0 + generated} algorithmic bytes per call\n")
            f.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=8) + "\n")
    cuda.close()


if __name__ == "__main__":
    main()
