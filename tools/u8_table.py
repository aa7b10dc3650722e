"""8-bit input frames: the fused 8-bit-in / 16-bit-out kernels and the 8-bit host-buffer calls, measured in one process with
CUDA events and host clocks around synchronising calls.  Writes <out-dir>/u8_table.jsonl, one JSON object per line:

  - kind "gpu": name, power limit and max SM clock of every visible GPU (nvidia-smi, read in the same run);
  - kind "kernel": every named mask / steering source x {f16, bf16} at 1080p x 64 and 4K x 32 frames (inputs resident in HBM,
    larger than L2), three launches interleaved round by round after a warm-up of each: the fp32-input 16-bit twin on the
    frames widened to float, the fused 8-bit kernel, and -- with --parent-lib, a build of the library before the fused 8-bit
    kernels existed -- that library's 8-bit launch of the same call (fp32 kernel into scratch + narrowing);
  - kind "e2e": the host-buffer calls with pinned frames and planes (cfg2 = G2/H2 on 64 x 1080p for M1 and M2, G4 steer at
    theta_d on 16 x 4K) at fp32 / f16 / bf16 planes, 8-bit frames against fp32 frames (and the parent library's fp32-frame
    call), each beside the copy ceiling of its own byte counts (plain cudaMemcpyAsync, one H2D and one D2H stream, as bench.py
    measures it), and the host time torch takes to widen the pinned 8-bit frames into pinned fp32 ones.

    python tools/u8_table.py [--out-dir DIR] [--parent-lib PATH] [--rounds 5] [--iters 10] [--skip kernel,e2e]"""
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
from cvsteer_b200 import capi  # noqa: E402
from cvsteer_b200.batch import G2Batch, G4Batch  # noqa: E402

DTYPES = [("f16", torch.float16), ("bf16", torch.bfloat16)]
FORMATS = [("f32", torch.float32)] + DTYPES
FMT = {torch.float32: capi.OUT_F32, torch.float16: capi.OUT_F16, torch.bfloat16: capi.OUT_BF16}
SC, MP, DOM = capi.STEER_SCALAR, capi.STEER_MAP, capi.STEER_DOMINANT
CASES = [("g2 M0 state", 2, capi.G2_MASK_STATE, DOM), ("g2 M1 orient", 2, capi.G2_MASK_ORIENT, DOM),
         ("g2 M2 full", 2, capi.G2_MASK_FULL, DOM), ("g2 lines", 2, capi.G2_MASK_LINES, DOM),
         ("g2 M2@scalar", 2, capi.G2_MASK_FULL, SC), ("g2 lines@scalar", 2, capi.G2_MASK_LINES, SC),
         ("g2 steer5@scalar", 2, capi.G2_MASK_STEER5, SC), ("g2 M2@map", 2, capi.G2_MASK_FULL, MP),
         ("g2 lines@map", 2, capi.G2_MASK_LINES, MP), ("g2 steer5@map", 2, capi.G2_MASK_STEER5, MP),
         ("g4 basis", 4, capi.G4_MASK_BASIS, DOM), ("g4 steer@map", 4, capi.G4_MASK_STEER, MP),
         ("g4 steer@scalar", 4, capi.G4_MASK_STEER, SC), ("g4 steer@theta_d", 4, capi.G4_MASK_STEER, DOM)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (v.strip() for v in l.split(","))))
            for l in q.stdout.strip().splitlines()]


def load_parent(path):
    """the other build of the library, with the signatures of the entry points it has"""
    l = C.CDLL(os.path.abspath(path))
    for name, (res, args) in capi._SIGS.items():
        fn = getattr(l, name, None)
        if fn is not None:
            fn.restype, fn.argtypes = res, args
    return l


class ParentHandle:
    def __init__(self, lib, family):
        self.lib, self.family, self.h = lib, family, C.c_void_p()
        width, spacing = (4, 0.67) if family == 2 else (6, 0.5)
        self.check(getattr(lib, f"cvs_g{family}_create")(C.byref(self.h), 0, width, spacing))

    def check(self, rc):
        if rc != 0:
            raise capi.CvsError(rc, self.lib.cvs_last_error().decode())

    def run_dev(self, x, mask, src, theta_map, outs, dt):
        n, rows, cols = x.shape
        es = torch.empty((), dtype=dt).element_size()
        arr = (C.c_void_p * (capi.G2_NPLANES if self.family == 2 else capi.G4_NPLANES))()
        for p, t in outs.items():
            arr[p] = t.data_ptr()
        b = capi.Batch()
        b.in_, b.in_is_u8, b.n, b.rows, b.cols = x.data_ptr(), int(x.dtype == torch.uint8), n, rows, cols
        b.in_pitch, b.in_frame_stride = x.stride(1) * x.element_size(), x.stride(0) * x.element_size()
        b.out_pitch, b.out_frame_stride = cols * es, rows * cols * es
        tm = C.c_void_p(theta_map.data_ptr()) if theta_map is not None else None
        fn = getattr(self.lib, f"cvs_g{self.family}_run_batch_dev_fmt")
        self.check(fn(self.h, C.byref(b), mask, src, 0.3, tm, arr, C.c_void_p(torch.cuda.current_stream().cuda_stream), FMT[dt]))

    def last_launch(self):
        name = C.create_string_buffer(96)
        self.check(self.lib.cvs_g2_last_launch(self.h, None, None, None, name, 96))
        return name.value.decode()

    def run_host_f32(self, xh, mask, src, outs, dt):
        n, rows, cols = xh.shape
        es = torch.empty((), dtype=dt).element_size()
        arr = (C.c_void_p * (capi.G2_NPLANES if self.family == 2 else capi.G4_NPLANES))()
        for p, t in outs.items():
            arr[p] = t.data_ptr()
        common = (C.c_void_p(xh.data_ptr()), n, rows, cols, cols * 4, rows * cols * 4, mask)
        tail = (arr, cols * es, rows * cols * es)
        if self.family == 2:
            self.check(self.lib.cvs_g2_run_batch_host_fmt(self.h, *common, *tail, FMT[dt]))
        else:
            self.check(self.lib.cvs_g4_run_batch_host_fmt(self.h, *common, src, 0.0, *tail, FMT[dt]))


def events_ms(fn, iters):
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def summary(v):
    return {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4)}


def kernels(a, emit, parent):
    for size, (n, rows, cols) in (("1080p", (64, 1080, 1920)), ("4k", (32, 2160, 3840))):
        x8 = torch.randint(0, 256, (n, rows, cols), dtype=torch.uint8, device="cuda")
        xf = x8.float()
        th = (torch.rand((n, rows, cols), device="cuda") - 0.5) * 3.1
        px = n * rows * cols
        hs = {2: G2Batch(), 4: G4Batch()}
        ph = {f: ParentHandle(parent, f) for f in (2, 4)} if parent is not None else {}
        for name, fam, mask, src in CASES:
            g = hs[fam]
            tm = th if src == MP else None
            kw = dict(steer=src, theta=0.3, theta_map=tm)
            for fname, dt in DTYPES:
                outs = {p: torch.empty((n, rows, cols), dtype=dt, device="cuda") for p in range(len(g._names)) if mask >> p & 1}
                runs = {"f32_in": lambda: g.run(xf, mask, outs=outs, out_dtype=dt, **kw),
                        "u8_fused": lambda: g.run(x8, mask, outs=outs, out_dtype=dt, **kw)}
                if fam in ph:
                    runs["u8_parent"] = lambda: ph[fam].run_dev(x8, mask, src, tm, outs, dt)
                names, times = {}, {k: [] for k in runs}
                for k, fn in runs.items():   # warm-up: module load, function attributes, tensor maps, scratch pool
                    fn()
                    fn()
                    names[k] = ph[fam].last_launch() if k == "u8_parent" else g.last_launch()["kernel"]
                torch.cuda.synchronize()
                for _ in range(a.rounds):
                    for k, fn in runs.items():
                        times[k].append(events_ms(fn, a.iters))
                nplanes = bin(mask).count("1")
                rec = {"kind": "kernel", "size": size, "frames": n, "case": name, "format": fname, "rounds": a.rounds,
                       "iters_per_round": a.iters, "B_px_f32_in": 4 + 2 * nplanes + (4 if src == MP else 0),
                       "B_px_u8_fused": 1 + 2 * nplanes + (4 if src == MP else 0)}
                for k in runs:
                    ms = statistics.median(times[k])
                    rec[k] = {"launched": names[k], **summary(times[k]), "Gpix_s": round(px / 1e9 / (ms / 1e3), 2)}
                med = {k: statistics.median(v) for k, v in times.items()}
                rec["u8_fused_vs_f32_in"] = round(med["f32_in"] / med["u8_fused"], 3)
                if "u8_parent" in med:
                    rec["u8_fused_vs_parent_fallback"] = round(med["u8_parent"] / med["u8_fused"], 3)
                emit(rec)
                del outs
        del x8, xf, th
        torch.cuda.empty_cache()


def pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype).pin_memory()


E2E = [("cfg2 M1", 2, capi.G2_MASK_ORIENT, (64, 1080, 1920)), ("cfg2 M2", 2, capi.G2_MASK_FULL, (64, 1080, 1920)),
       ("g4 steer@theta_d 4k", 4, capi.G4_MASK_STEER, (16, 2160, 3840))]


def e2e(a, emit, parent):
    for name, fam, mask, (n, rows, cols) in E2E:
        px = n * rows * cols
        g = G2Batch() if fam == 2 else G4Batch()
        pg = ParentHandle(parent, fam) if parent is not None else None
        planes = [p for p in range(len(g._names)) if mask >> p & 1]
        xh8 = pinned((n, rows, cols), torch.uint8)
        xh8.copy_(torch.randint(0, 256, (n, rows, cols), dtype=torch.uint8))
        xh32 = pinned((n, rows, cols), torch.float32)
        widen = []
        for _ in range(a.rounds + 1):   # what a caller with 8-bit frames does today before the fp32 call
            t0 = time.perf_counter()
            xh32.copy_(xh8)
            widen.append(time.perf_counter() - t0)
        widen = widen[1:]
        emit({"kind": "widen", "config": name, "frames": n, "bytes_written": px * 4, "rounds": a.rounds,
              "ms_median": round(statistics.median(widen) * 1e3, 2), "ms_min": round(min(widen) * 1e3, 2),
              "ms_max": round(max(widen) * 1e3, 2), "api": "torch: pinned_fp32.copy_(pinned_u8)"})
        dev_in = {torch.uint8: torch.empty((n, rows, cols), dtype=torch.uint8, device="cuda"),
                  torch.float32: torch.empty((n, rows, cols), device="cuda")}
        for fname, dt in FORMATS:
            es = torch.empty((), dtype=dt).element_size()
            outs = {p: pinned((n, rows, cols), dt) for p in planes}
            dev_out = [torch.empty((n, rows, cols), dtype=dt, device="cuda") for _ in planes]
            kw = {} if fam == 2 else {"theta": None}
            runs = {"u8_in": lambda: g.run_host(xh8, mask, outs, **kw), "f32_in": lambda: g.run_host(xh32, mask, outs, **kw)}
            if pg is not None:
                runs["f32_in_parent"] = lambda: pg.run_host_f32(xh32, mask, DOM, outs, dt)
            ins = {"u8_in": xh8, "f32_in": xh32, "f32_in_parent": xh32}
            s_h2d, s_d2h = torch.cuda.Stream(), torch.cuda.Stream()

            def ceiling(xh):
                with torch.cuda.stream(s_h2d):
                    dev_in[xh.dtype].copy_(xh, non_blocking=True)
                with torch.cuda.stream(s_d2h):
                    for i, p in enumerate(planes):
                        outs[p].copy_(dev_out[i], non_blocking=True)
                s_h2d.synchronize()
                s_d2h.synchronize()

            res = {k: {"run": [], "ceil": []} for k in runs}
            for k, fn in runs.items():   # warm-up: staging ring, handles, pinned pages
                fn()
                ceiling(ins[k])
            for _ in range(a.rounds):
                for k, fn in runs.items():
                    t0 = time.perf_counter()
                    fn()
                    res[k]["run"].append(time.perf_counter() - t0)
                    t0 = time.perf_counter()
                    ceiling(ins[k])
                    res[k]["ceil"].append(time.perf_counter() - t0)
            rec = {"kind": "e2e", "config": name, "frames": n, "rows": rows, "cols": cols, "format": fname, "gpus": 1,
                   "rounds": a.rounds, "d2h_bytes": px * es * len(planes)}
            for k in runs:
                h2d = px * (1 if k == "u8_in" else 4)
                run, ceil = statistics.median(res[k]["run"]), statistics.median(res[k]["ceil"])
                rec[k] = {"h2d_bytes": h2d, "B_px": h2d // px + es * len(planes), "ms_median": round(run * 1e3, 2),
                          "ms_min": round(min(res[k]["run"]) * 1e3, 2), "ms_max": round(max(res[k]["run"]) * 1e3, 2),
                          "Mpix_s": round(px / 1e6 / run, 1), "ceiling_ms": round(ceil * 1e3, 2),
                          "ceiling_Mpix_s": round(px / 1e6 / ceil, 1), "frac_of_ceiling": round(ceil / run, 3)}
            rec["u8_vs_f32_in"] = round(rec["f32_in"]["ms_median"] / rec["u8_in"]["ms_median"], 3)
            if pg is not None:
                rec["f32_in_vs_parent"] = round(rec["f32_in_parent"]["ms_median"] / rec["f32_in"]["ms_median"], 3)
            emit(rec)
            del outs, dev_out
        del xh8, xh32, dev_in, g, pg
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default="u8_table")
    ap.add_argument("--parent-lib", default=None, help="a build of the library without the fused 8-bit kernels, for the "
                                                        "fallback it ran and its fp32-frame host path")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--skip", default="", help="comma list of parts to skip: kernel, e2e")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("u8_table needs a CUDA device")
    parent = load_parent(a.parent_lib) if a.parent_lib else None
    os.makedirs(a.out_dir, exist_ok=True)
    path = os.path.join(a.out_dir, "u8_table.jsonl")
    with open(path, "w") as fh:
        def emit(r):
            fh.write(json.dumps(r) + "\n")
            fh.flush()
            print(json.dumps(r), flush=True)
        for gpu in gpu_info():
            emit({"kind": "gpu", **gpu})
        if "kernel" not in a.skip:
            kernels(a, emit, parent)
        if "e2e" not in a.skip:
            e2e(a, emit, parent)


if __name__ == "__main__":
    main()
