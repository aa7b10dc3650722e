"""fp32 against 16-bit (fp16 / bf16) output planes, measured in one process with CUDA events and host clocks around
synchronising calls.  Writes <out-dir>/out16_table.jsonl, one JSON object per line:

  - kind "gpu": name, power limit and max SM clock of every visible GPU (nvidia-smi, read in the same run);
  - kind "kernel": every named mask / steering source at 1080p x 64 and 4K x 32 frames (inputs resident in HBM, larger than
    L2), the three formats interleaved round by round after a warm-up of each; Gpix/s, and the fraction of the binding
    roofline from the format's own byte count (4 B in + 4 or 2 B per output plane + 4 B per angle-map pixel) and the
    fp32 instruction count of tools/kernel_table.py;
  - kind "e2e": cfg2 (G2/H2 M2 on 1080p frames) through the host-buffer call, pinned host planes of each format, beside the
    copy ceiling of its own byte counts (plain cudaMemcpyAsync: one H2D and one D2H stream per GPU, as bench.py measures
    it), on 1 GPU and over every GPU (cvs_g2_run_batch_host_multi[_fmt]).

    python tools/out16_table.py [--out-dir DIR] [--rounds 5] [--iters 10] [--e2e-frames 64] [--multi-frames 16]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from cvsteer_b200 import capi  # noqa: E402
from cvsteer_b200.batch import G2Batch, G4Batch  # noqa: E402
from kernel_table import FP32_NOMINAL, hbm_peak  # noqa: E402

FORMATS = [("f32", torch.float32), ("f16", torch.float16), ("bf16", torch.bfloat16)]
SC, MP, DOM = capi.STEER_SCALAR, capi.STEER_MAP, capi.STEER_DOMINANT
# name, family, mask, steering source, fp32 instructions per pixel (tools/kernel_table.py)
CASES = [("g2 M0 state", 2, capi.G2_MASK_STATE, DOM, 167), ("g2 M1 orient", 2, capi.G2_MASK_ORIENT, DOM, 167),
         ("g2 M2 full", 2, capi.G2_MASK_FULL, DOM, 217), ("g2 lines", 2, capi.G2_MASK_LINES, DOM, 217),
         ("g2 M2@scalar", 2, capi.G2_MASK_FULL, SC, 217), ("g2 lines@scalar", 2, capi.G2_MASK_LINES, SC, 217),
         ("g2 steer5@scalar", 2, capi.G2_MASK_STEER5, SC, 199), ("g2 M2@map", 2, capi.G2_MASK_FULL, MP, 227),
         ("g2 lines@map", 2, capi.G2_MASK_LINES, MP, 227), ("g2 steer5@map", 2, capi.G2_MASK_STEER5, MP, 209),
         ("g4 basis", 4, capi.G4_MASK_BASIS, DOM, 273), ("g4 steer@map", 4, capi.G4_MASK_STEER, MP, 323),
         ("g4 steer@scalar", 4, capi.G4_MASK_STEER, SC, 313), ("g4 steer@theta_d", 4, capi.G4_MASK_STEER, DOM, 393)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (v.strip() for v in l.split(","))))
            for l in q.stdout.strip().splitlines()]


def events_ms(fn, iters):
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels(a, emit):
    hbm = hbm_peak()
    for size, (n, rows, cols) in (("1080p", (64, 1080, 1920)), ("4k", (32, 2160, 3840))):
        x = torch.rand((n, rows, cols), device="cuda") * 255
        th = (torch.rand((n, rows, cols), device="cuda") - 0.5) * 3.1
        px = n * rows * cols
        g2, g4 = G2Batch(), G4Batch()
        for name, fam, mask, src, ipp in CASES:
            g = g2 if fam == 2 else g4
            nplanes = bin(mask).count("1")
            kw = dict(steer=src, theta=0.3, theta_map=th if src == MP else None)
            outs = {f: {p: torch.empty((n, rows, cols), dtype=dt, device="cuda") for p in range(len(g._names)) if mask >> p & 1}
                    for f, dt in FORMATS}
            names, times = {}, {f: [] for f, _ in FORMATS}
            for f, dt in FORMATS:   # warm-up: module load, function attributes, tensor maps
                for _ in range(2):
                    g.run(x, mask, outs=outs[f], out_dtype=dt, **kw)
                names[f] = g.last_launch()["kernel"]
            torch.cuda.synchronize()
            for _ in range(a.rounds):
                for f, dt in FORMATS:
                    times[f].append(events_ms(lambda: g.run(x, mask, outs=outs[f], out_dtype=dt, **kw), a.iters))
            for f, dt in FORMATS:
                ms = statistics.median(times[f])
                bpp = 4 + nplanes * (4 if dt == torch.float32 else 2) + (4 if src == MP else 0)
                gpix = px / 1e9 / (ms / 1e3)
                t_h, t_f = px * bpp / (hbm * 1e9), px * ipp / FP32_NOMINAL
                emit({"kind": "kernel", "size": size, "frames": n, "case": name, "format": f, "launched": names[f],
                      "ms_median": round(ms, 4), "ms_min": round(min(times[f]), 4), "ms_max": round(max(times[f]), 4),
                      "rounds": a.rounds, "iters_per_round": a.iters, "Gpix_s": round(gpix, 2), "B_px": bpp, "instr_px_fp32": ipp,
                      "binding": "fp32" if t_f > t_h else "hbm", "frac_of_binding": round(max(t_h, t_f) / (ms / 1e3), 3),
                      "hbm_GBs_used": hbm})
            del outs
        del x, th
        torch.cuda.empty_cache()


def pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype).pin_memory()


def e2e(a, emit):
    rows, cols, mask = 1080, 1920, capi.G2_MASK_FULL
    planes = [p for p in range(capi.G2_NPLANES) if mask >> p & 1]
    ndev = torch.cuda.device_count()
    lib = capi.lib()
    for world, per in [(1, a.e2e_frames)] + ([(ndev, a.multi_frames)] if ndev > 1 else []):
        n = world * per
        px = n * rows * cols
        xh = pinned((n, rows, cols), torch.float32)
        xh.copy_(torch.rand((n, rows, cols)) * 255)
        hosts = {f: {p: pinned((n, rows, cols), dt) for p in planes} for f, dt in FORMATS}
        # device copies for the ceiling: `per` frames per GPU, the same byte counts as the pipeline moves
        dev_in = [torch.empty((per, rows, cols), device=f"cuda:{d}") for d in range(world)]
        dev_out = {f: [[torch.empty((per, rows, cols), dtype=dt, device=f"cuda:{d}") for _ in planes] for d in range(world)]
                   for f, dt in FORMATS}
        g = G2Batch(device=0)

        def run(f, dt):
            if world == 1:
                g.run_host(xh, mask, hosts[f])
                return
            arr = (C.c_void_p * capi.G2_NPLANES)()
            for p in planes:
                arr[p] = hosts[f][p].data_ptr()
            es = 4 if dt == torch.float32 else 2
            common = (world, None, 4, 0.67, C.c_void_p(xh.data_ptr()), n, rows, cols, cols * 4, rows * cols * 4, mask, arr,
                      cols * es, rows * cols * es)
            capi.check(lib.cvs_g2_run_batch_host_multi(*common) if dt == torch.float32 else
                       lib.cvs_g2_run_batch_host_multi_fmt(*common, capi.OUT_F16 if dt == torch.float16 else capi.OUT_BF16))

        def ceiling(f):
            streams = [(torch.cuda.Stream(device=d), torch.cuda.Stream(device=d)) for d in range(world)]
            for d in range(world):
                lo = d * per
                with torch.cuda.stream(streams[d][0]):
                    dev_in[d].copy_(xh[lo:lo + per], non_blocking=True)
                with torch.cuda.stream(streams[d][1]):
                    for i, p in enumerate(planes):
                        hosts[f][p][lo:lo + per].copy_(dev_out[f][d][i], non_blocking=True)
            for s1, s2 in streams:
                s1.synchronize()
                s2.synchronize()

        res = {f: {"run": [], "ceil": []} for f, _ in FORMATS}
        for f, dt in FORMATS:   # warm-up: staging ring, handles, pinned pages
            run(f, dt)
            ceiling(f)
        for _ in range(a.rounds):
            for f, dt in FORMATS:
                t0 = time.perf_counter()
                run(f, dt)
                res[f]["run"].append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                ceiling(f)
                res[f]["ceil"].append(time.perf_counter() - t0)
        for f, dt in FORMATS:
            es = 4 if dt == torch.float32 else 2
            h2d, d2h = px * 4, px * es * len(planes)
            dt_run, dt_ceil = statistics.median(res[f]["run"]), statistics.median(res[f]["ceil"])
            emit({"kind": "e2e", "config": "cfg2 M2 1080p", "gpus": world, "frames": n, "format": f,
                  "api": "cvs_g2_run_batch_host" + ("_multi" if world > 1 else "") + ("" if f == "f32" else "_fmt"),
                  "B_px": 4 + es * len(planes), "h2d_bytes": h2d, "d2h_bytes": d2h, "rounds": a.rounds,
                  "ms_median": round(dt_run * 1e3, 2), "Mpix_s": round(px / 1e6 / dt_run, 1),
                  "GB_s": round((h2d + d2h) / 1e9 / dt_run, 1), "ceiling_GB_s": round((h2d + d2h) / 1e9 / dt_ceil, 1),
                  "ceiling_Mpix_s": round(px / 1e6 / dt_ceil, 1), "frac_of_ceiling": round(dt_ceil / dt_run, 3)})
        del xh, hosts, dev_in, dev_out, g
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default="out16_table")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--e2e-frames", type=int, default=64)
    ap.add_argument("--multi-frames", type=int, default=16, help="frames per GPU of the all-GPU end-to-end row")
    ap.add_argument("--skip", default="", help="comma list of parts to skip: kernel, e2e")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("out16_table needs a CUDA device")
    os.makedirs(a.out_dir, exist_ok=True)
    path = os.path.join(a.out_dir, "out16_table.jsonl")
    with open(path, "w") as fh:
        def emit(r):
            fh.write(json.dumps(r) + "\n")
            fh.flush()
            print(json.dumps(r), flush=True)
        for gpu in gpu_info():
            emit({"kind": "gpu", **gpu})
        if "kernel" not in a.skip:
            kernels(a, emit)
        if "e2e" not in a.skip:
            e2e(a, emit)


if __name__ == "__main__":
    main()
