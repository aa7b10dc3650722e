#!/usr/bin/env python
"""Contract benchmark for the cvsteer hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode M0|M1|M2]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline: a "step" is one pass of the fused G2/H2 basis+steer+orientation kernel over one batch of synthetic frames
(BASELINE.json configs[1]: 64 frames of 1920x1080 per GPU, fp32, single scale) already resident in HBM.  Rank 0 prints
ONE JSON line.  See DESIGN.md "Measurement" for how every field is derived.

  value      whole-job Mpix/s, device-timed (CUDA events on the launching stream, max over ranks), exactly K steps
  roofline   the BINDING side of the kernel's roofline: algorithmic bytes / measured launch duration against the measured
             HBM copy rate (MEASURED_PEAKS.json), or algorithmic fp32 instructions against the nominal issue rate
             148 SM x 128 lanes x 1.965 GHz = 37.2 T instr/s -- whichever bound is slower; both sides, the FFMA
             microbenchmark measured in the same process, and a >= 2 s sustained run (power-capped clocks) are reported
  e2e        the same metric through the host-buffer C-ABI call (cvs_g2_run_batch_host): pinned host frames in, pinned
             host planes out, H2D + D2H inside the timed region; with the PCIe ceiling of the same byte counts (plain
             concurrent copies, all ranks at once) measured beside it
  cpu_baseline  the oracle (the reference's glue over the same OpenCV primitives, cv2) on this box's host cores,
             frame-parallel like the reference's cv::parallel_for_ (example/steer.cpp:169), bounded sample
  configs    the other BASELINE.json configurations, each with its own roofline and clocks: 4K frames in modes M0/M1/M2
             (the north-star target size), cfg3 (5-level pyramid, 256 4K frames in total: strong scaling over N), cfg4
             (G4/H4 steer at an angle map + phase, 256 4K frames in total), cfg5 (one 32768^2 image in row bands: compute
             only / NCCL gather / compute+gather fused over peer memory)

--impl reference runs only that CPU path and prints the same line shape with "impl": "reference".
--cfg1 measures BASELINE.json configs[0] instead (the cvsteer-run per-file body on the bundled test image).
--dump-outputs DIR writes, after the K timed steps, what the last one computed: DIR/<plane>.npy (float32) for every output plane
of the headline launch, each at the same 2^20 pixels of the 64-frame batch (flat indices drawn by np.random.default_rng(0),
sorted).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS, COLS, FRAMES = 1080, 1920, 64          # BASELINE.json configs[1]
WORKLOAD = "cfg2: G2/H2 (width 4, spacing 0.67) on 64 synthetic 1920x1080 fp32 frames per GPU, single scale"
# algorithmic bytes / fp32 instructions per pixel per mode (SURVEY.md section 8d; DESIGN.md "Roofline")
MODES = {
    "M0": dict(bpp=52, ipp=167, what="materialise class state: 7 basis planes + c1..c3 + theta_d + strength"),
    "M1": dict(bpp=16, ipp=167, what="orientation: theta_d, strength, energy at theta_d"),
    "M2": dict(bpp=32, ipp=217, what="basis+steer+orientation: theta_d, strength, g2, h2, e, magnitude, phase"),
}
FP32_NOMINAL = 148 * 128 * 1.965e9           # fp32 instructions/s: 148 SMs x 128 lanes x max SM clock
PYR5 = sum(0.25 ** l for l in range(5))      # pixels of a 5-level pyramid per level-0 pixel (1.332)
DUMP_PIXELS = 1 << 20                        # --dump-outputs: sampled pixels per plane (12 planes at most: 48 MB in all)


def env_int(k, d):
    return int(os.environ.get(k, d))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU reference arm (oracle over cv2), frame-parallel
# ------------------------------------------------------------------------------------------------
def _cpu_frames(n, seed0):
    import numpy as np
    return [np.random.default_rng(seed0 + i).uniform(0, 255, (ROWS, COLS)).astype(np.float32) for i in range(n)]


def _cpu_one(mode, img):
    from oracle import cvsteer_ref as ref
    if mode == "M2":
        ref.g2_full(img)            # ctor + steer(theta_d map, g2,h2,e,magnitude,phase): what both reference callers run
    elif mode == "M1":
        ref.g2_orientation(img)
    else:
        ref.SteerableFiltersG2(img)


def cpu_pass(mode, frames, workers):
    """One frame-parallel pass; returns seconds."""
    from concurrent.futures import ThreadPoolExecutor
    t0 = time.perf_counter()
    with ThreadPoolExecutor(workers) as ex:
        list(ex.map(lambda f: _cpu_one(mode, f), frames))
    return time.perf_counter() - t0


def cpu_setup():
    import cv2
    cv2.setNumThreads(1)            # one worker thread per core, OpenCV single-threaded inside each (SURVEY 8d)
    cores = os.cpu_count() or 1
    workers = min(cores, 64)
    return cores, workers


def cpu_baseline(mode):
    cores, workers = cpu_setup()
    nframes = max(16, 2 * workers)
    nframes = min(nframes, 96)
    frames = _cpu_frames(nframes, 2000)
    cpu_pass(mode, frames[:workers], workers)          # warm-up
    dt = cpu_pass(mode, frames, workers)
    return {"value": round(nframes * ROWS * COLS / 1e6 / dt, 2), "unit": "Mpix/s", "cores": workers, "kind": "port",
            "sample": f"{nframes} of the workload's 1920x1080 frames, mode {mode}, {workers} frame-parallel threads "
                      f"(host has {cores} logical cores), cv2.setNumThreads(1), 1 warm-up pass"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores, workers = cpu_setup()
    per_step = max(8, workers)
    per_step = min(per_step, 64)
    frames = _cpu_frames(per_step, 2000)
    for _ in range(args.warmup):
        cpu_pass(args.mode, frames, workers)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_pass(args.mode, frames, workers)
    dt = (time.perf_counter() - t0) / args.steps
    val = round(per_step * ROWS * COLS / 1e6 / dt, 2)
    sample = (f"each step = {per_step} of the workload's 64 frames, {workers} frame-parallel threads "
              f"(host has {cores} logical cores), cv2.setNumThreads(1)")
    line = {"impl": "reference", "metric": "G2/H2 basis+steer throughput", "value": val, "unit": "Mpix/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "mode": args.mode, "what": MODES[args.mode]["what"],
                       "arm": "oracle/cvsteer_ref.py: the reference's glue over cv2 (the reference C++ cannot be "
                              "built here: no OpenCV C++ headers)"},
            "cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": workers, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler (NVML, polled during the timed regions)
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.stop_flag, self.ok = [], False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.004)

    def summary(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        nv = self.nv
        win = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-5:]
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        bits = 0
        for s in win:
            bits |= s[2]
        return {"sm_mhz": statistics.median(s[1] for s in win) if win else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(v for k, v in names.items() if bits & k), "samples": len(win)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    """Per-process state shared by the config runners."""

    def __init__(self, rank, local_rank, world):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.local, self.world = rank, local_rank, world
        self.dev = torch.device("cuda", local_rank)
        self.hbm_peak, self.peak_src = load_peaks()
        self.sampler = ClockSampler(local_rank)
        self.fp32_measured = None     # T instr/s, FFMA microbenchmark (rank 0)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warm):
        """W untimed calls, barrier, K timed calls between CUDA events on the launching stream, barrier; max over ranks.
        Returns (ms per step, clocks summary of the timed window)."""
        torch = self.torch
        for _ in range(warm):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        t1 = time.perf_counter()
        ms = self.max_over_ranks(e0.elapsed_time(e1) / steps)
        return ms, self.sampler.summary(t0, t1)

    def roofline(self, px, bpp, ipp, ms, kernel=None, traffic=None, sustained=None, brief=True):
        """Both sides of the roofline for `px` pixels per launch in `ms`; the top-level keys describe the BINDING side.
        brief: leave out the prose (how each denominator was obtained) -- the headline's roofline carries it once."""
        gbs = px * bpp / 1e9 / (ms / 1e3)
        tis = px * ipp / 1e12 / (ms / 1e3)
        t_h, t_f = px * bpp / (self.hbm_peak * 1e9), px * ipp / FP32_NOMINAL
        hbm = {"achieved_GB_s": round(gbs, 1), "peak_GB_s": self.hbm_peak, "frac": round(gbs / self.hbm_peak, 3),
               "peak_source": self.peak_src}
        fp = {"achieved_Tinstr_s": round(tis, 2), "peak_Tinstr_s_nominal": round(FP32_NOMINAL / 1e12, 2),
              "frac_of_nominal": round(tis * 1e12 / FP32_NOMINAL, 3),
              "nominal_how": "148 SMs x 128 fp32 lanes x 1.965 GHz max SM clock (fixed ceiling)"}
        if self.fp32_measured:
            fp["peak_Tinstr_s_measured"] = round(self.fp32_measured, 2)
            fp["frac_of_measured"] = round(tis / self.fp32_measured, 3)
            fp["measured_how"] = ("cvs_bench_ffma in this process: 512 immediate-operand FFMAs per loop trip, 16 warps per "
                                  "scheduler; floats with the power state, so the nominal figure is the denominator of `frac`")
        r = {"bound": "fp32" if t_f > t_h else "hbm"}
        if t_f > t_h:
            r.update({"achieved": round(tis, 2), "peak": round(FP32_NOMINAL / 1e12, 2), "unit": "T fp32 instr/s",
                      "frac": round(tis * 1e12 / FP32_NOMINAL, 3), "peak_source": "nominal issue rate at max SM clock"})
        else:
            r.update({"achieved": round(gbs, 1), "peak": self.hbm_peak, "unit": "GB/s", "frac": round(gbs / self.hbm_peak, 3),
                      "peak_source": self.peak_src})
        r.update({"traffic": traffic, "algorithmic_bytes_per_px": bpp, "algorithmic_fp32_instr_per_px": ipp,
                  "px_per_launch": px, "kernel_ms": round(ms, 4), "hbm": hbm, "fp32": fp})
        if kernel:
            r["kernel"] = kernel
        if sustained:
            r["sustained"] = sustained
        if brief:
            for d in (r, hbm, fp):
                for k in ("peak_source", "nominal_how", "measured_how"):
                    d.pop(k, None)
        return r


def traffic_of(mode):
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tp)).get(mode)
    except Exception:
        return None


def run_headline(cx, args):
    """cfg2: K steps of the fused kernel over 64 resident 1080p frames per GPU (weak scaling), + a >= 2 s sustained run."""
    torch = cx.torch
    from cvsteer_b200 import capi
    from cvsteer_b200.batch import G2Batch
    mode = args.mode
    mask = {"M0": capi.G2_MASK_STATE, "M1": capi.G2_MASK_ORIENT, "M2": capi.G2_MASK_FULL}[mode]
    planes = [p for p in range(capi.G2_NPLANES) if mask >> p & 1]
    px = FRAMES * ROWS * COLS
    gen = torch.Generator(device=cx.dev)
    gen.manual_seed(2000 + cx.rank)
    x = torch.rand((FRAMES, ROWS, COLS), device=cx.dev, generator=gen) * 255.0       # 531 MB > 126 MB L2
    outs = {p: torch.empty((FRAMES, ROWS, COLS), device=cx.dev) for p in planes}
    g = G2Batch(device=cx.local)
    lib = capi.lib()
    for _ in range(max(args.warmup, 3)):
        g.run(x, mask, outs=outs)
    cx.barrier()
    l0 = lib.cvs_launch_count()
    ms, clocks = cx.timed(lambda: g.run(x, mask, outs=outs), args.steps, 0)
    launches = lib.cvs_launch_count() - l0
    launch = g.last_launch()
    value = cx.world * px / 1e6 / (ms / 1e3)
    dump = output_sample(cx, outs, planes) if args.dump_outputs and cx.rank == 0 else None

    # sustained: the same launch back to back for >= 2 s (the power cap pulls the SM clock down after a few hundred ms)
    sustained = None
    if not args.quick:
        n_sus = max(args.steps, int(args.sustain_s * 1e3 / ms) + 1)
        ms_s, clk_s = cx.timed(lambda: g.run(x, mask, outs=outs), n_sus, 0)
        sustained = {"seconds": round(n_sus * ms_s / 1e3, 2), "launches": n_sus, "kernel_ms": round(ms_s, 4),
                     "Mpix_s": round(cx.world * px / 1e6 / (ms_s / 1e3), 1),
                     "frac_fp32_nominal": round(px * MODES[mode]["ipp"] / (ms_s / 1e3) / FP32_NOMINAL, 3),
                     "frac_hbm_measured": round(px * MODES[mode]["bpp"] / 1e9 / (ms_s / 1e3) / cx.hbm_peak, 3), "clocks": clk_s}
    roof = cx.roofline(px, MODES[mode]["bpp"], MODES[mode]["ipp"], ms, launch["kernel"], traffic_of(mode), sustained, brief=False)
    cfg = {"workload": WORKLOAD, "mode": mode, "what": MODES[mode]["what"], "frames_per_gpu": FRAMES, "rows": ROWS,
           "cols": COLS, "sharding": "frames, no collective",
           "l2": "inputs (531 MB/GPU) larger than the 126 MB L2; no flush needed",
           "grid": launch["grid"], "block": launch["block"], "smem": launch["smem"]}
    return dict(value=value, ms=ms, clocks=clocks, launches=int(launches), roofline=roof, config=cfg,
                state=(g, x, outs, mask, planes, px), dump=dump)


def output_sample(cx, outs, planes):
    """The headline planes as they are now (after the last timed step) at DUMP_PIXELS fixed, seeded positions of the batch."""
    import numpy as np
    from cvsteer_b200 import capi
    px = FRAMES * ROWS * COLS
    idx = np.sort(np.random.default_rng(0).choice(px, min(px, DUMP_PIXELS), replace=False))
    assert idx.size * 4 * len(planes) <= 64 << 20
    idx = cx.torch.from_numpy(idx).to(cx.dev)
    return {capi.G2_PLANE_NAMES[p]: outs[p].view(-1)[idx].cpu().numpy() for p in planes}


def write_dump(d, arrays):
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a, np.float32))


def run_e2e(cx, args, state):
    """The host-buffer C-ABI call with pinned host memory allocated on the GPU's NUMA node, and the PCIe ceiling of the
    same byte counts (one plain H2D + one plain D2H stream, all ranks at once) beside it."""
    torch = cx.torch
    from cvsteer_b200 import hostmem
    g, x, outs, mask, planes, px = state
    old_aff = os.sched_getaffinity(0)
    numa = hostmem.bind_to_gpu_numa(cx.local) if not args.no_numa else {"node": None, "cpus": 0, "bound": False}
    try:
        xh = torch.empty((FRAMES, ROWS, COLS), dtype=torch.float32).pin_memory()
        xh.copy_(x)
        oh = {p: torch.empty((FRAMES, ROWS, COLS), dtype=torch.float32).pin_memory() for p in planes}
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        g.run_host(xh, mask, oh)                                   # warm-up (allocates the device staging ring)
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            g.run_host(xh, mask, oh)                               # synchronous: returns when results are in host memory
        dt = cx.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
        chk = float(oh[planes[0]][0, 100, 100])                    # touch a result on the host
        h2d, d2h = px * 4, px * 4 * len(planes)
        # ceiling: the same bytes as plain copies, both directions concurrently, all ranks at once
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        dsrc = [outs[p] for p in planes]
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            with torch.cuda.stream(s1):
                x.copy_(xh, non_blocking=True)
            with torch.cuda.stream(s2):
                for p, d in zip(planes, dsrc):
                    oh[p].copy_(d, non_blocking=True)
            s1.synchronize()
            s2.synchronize()
        dt_c = cx.max_over_ranks((time.perf_counter() - t0) / 2)
        e2e = {"value": round(cx.world * px / 1e6 / dt, 1), "unit": "Mpix/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": round(dt * 1e3, 2),
               "api": "cvs_g2_run_batch_host (pinned host buffers, 3-stage H2D/kernel/D2H pipeline)",
               "achieved_GB_s_per_gpu": round((h2d + d2h) / 1e9 / dt, 1),
               "pcie_ceiling_gbs": round(cx.world * (h2d + d2h) / 1e9 / dt_c, 1),
               "pcie_ceiling_how": "the same H2D + D2H byte counts as plain cudaMemcpyAsync on two streams, all ranks "
                                   "concurrently, pinned memory on the GPU's NUMA node; whole-job GB/s",
               "frac_of_ceiling": round(dt_c / dt, 3), "numa": numa, "probe": chk}
        del xh, oh
        return e2e
    finally:
        try:
            os.sched_setaffinity(0, old_aff)
        except Exception:
            pass


def run_4k_modes(cx, args):
    """The north-star target size: 32 resident 3840x2160 frames per GPU (1.06 GB in), every mode, kernel only."""
    torch = cx.torch
    from cvsteer_b200 import capi
    from cvsteer_b200.batch import G2Batch
    n, R, C = 32, 2160, 3840
    px = n * R * C
    x = torch.rand((n, R, C), device=cx.dev) * 255.0
    g = G2Batch(device=cx.local)
    res = {}
    steps = max(5, min(args.steps, 20))
    for m, mk in (("M0", capi.G2_MASK_STATE), ("M1", capi.G2_MASK_ORIENT), ("M2", capi.G2_MASK_FULL)):
        o = {p: torch.empty((n, R, C), device=cx.dev) for p in range(capi.G2_NPLANES) if mk >> p & 1}
        ms, clk = cx.timed(lambda: g.run(x, mk, outs=o), steps, 3)
        res["4k_" + m] = {"workload": f"G2/H2 mode {m} on {n} synthetic 3840x2160 frames per GPU, single scale, kernel only",
                          "scaling": "weak", "steps": steps, "ms_per_step": round(ms, 4),
                          "Mpix_s": round(cx.world * px / 1e6 / (ms / 1e3), 1),
                          "roofline": cx.roofline(px, MODES[m]["bpp"], MODES[m]["ipp"], ms, g.last_launch()["kernel"]), "clocks": clk}
        del o
    del x
    torch.cuda.empty_cache()
    return res


def run_cfg3(cx, args):
    """configs[2]: G2/H2 orientation (M1) over a 5-level pyramid, 256 4K frames IN TOTAL, sharded by frame (strong)."""
    torch = cx.torch
    from cvsteer_b200 import capi, multi
    from cvsteer_b200.batch import G2Batch
    total, R, C, L = args.frames_total, 2160, 3840, 5
    lo, hi = multi.shard_frames(total, cx.world, cx.rank)
    n = hi - lo
    x = torch.rand((n, R, C), device=cx.dev) * 255.0
    g = G2Batch(device=cx.local)
    shapes = [(R, C)]
    for _ in range(L - 1):
        shapes.append(((shapes[-1][0] + 1) // 2, (shapes[-1][1] + 1) // 2))
    outs = [{p: torch.empty((n,) + s, device=cx.dev) for p in (capi.THETA, capi.STRENGTH, capi.E)} for s in shapes]
    lv = [x] + [torch.empty((n,) + s, device=cx.dev) for s in shapes[1:]]   # every level stays resident

    def step():   # one launch per level: the fused kernel also emits the next level from the tile it has staged
        for l in range(L):
            g.run(lv[l], capi.G2_MASK_ORIENT, outs=outs[l], next_level=lv[l + 1] if l + 1 < L else None)
    steps = max(3, min(args.steps, 10))
    ms, clk = cx.timed(step, steps, 2)
    px0 = total * R * C
    # per level-0 pixel: every level reads its input once and writes 3 planes (16 B x 1.332); levels 1..4 are also
    # written once by the level above (4 B x 0.332); 167 instructions per pixel of every level + ~4 per emitted pixel
    bpp, ipp = 16 * PYR5 + 4 * (PYR5 - 1), 167 * PYR5 + 4 * (PYR5 - 1)
    r = {"workload": f"cfg3: G2/H2 M1 over a 5-level pyramid, {total} synthetic 3840x2160 frames in total, "
                     f"{n} on this GPU, every level resident", "scaling": "strong", "collective": "none (frames are independent)",
         "steps": steps, "launches_per_step": L, "ms_per_step": round(ms, 3), "Mpix_s_level0": round(px0 / 1e6 / (ms / 1e3), 1),
         "roofline": cx.roofline(px0 // cx.world, round(bpp, 2), round(ipp, 1), ms, g.last_launch()["kernel"] + " x5 levels"),
         "clocks": clk}
    del x, outs, lv
    torch.cuda.empty_cache()
    return r


def run_cfg4(cx, args):
    """configs[3]: G4/H4 steer at a per-pixel angle map (+ magnitude, phase), 256 4K frames in total, sharded by frame."""
    torch = cx.torch
    from cvsteer_b200 import capi, multi
    from cvsteer_b200.batch import G2Batch, G4Batch
    total, R, C = args.frames_total, 2160, 3840
    lo, hi = multi.shard_frames(total, cx.world, cx.rank)
    n = hi - lo
    x = torch.rand((n, R, C), device=cx.dev) * 255.0
    g2, g4 = G2Batch(device=cx.local), G4Batch(device=cx.local)
    th = g2.run(x, capi.bit(capi.THETA))["theta"]          # precomputed, resident theta_d of the same frames (SURVEY 8d)
    outs = {p: torch.empty((n, R, C), device=cx.dev) for p in (capi.G4T, capi.H4T, capi.MAG4, capi.PHASE4)}
    steps = max(3, min(args.steps, 10))
    ms, clk = cx.timed(lambda: g4.run(x, capi.G4_MASK_STEER, steer=capi.STEER_MAP, theta_map=th, outs=outs), steps, 2)
    px0 = total * R * C
    r = {"workload": f"cfg4: G4/H4 steer(theta map) + magnitude + phase, {total} synthetic 3840x2160 frames in total, "
                     f"{n} on this GPU", "scaling": "strong", "collective": "none (frames are independent)", "steps": steps,
         "ms_per_step": round(ms, 3), "Mpix_s": round(px0 / 1e6 / (ms / 1e3), 1),
         "roofline": cx.roofline(px0 // cx.world, 24, 323, ms, g4.last_launch()["kernel"]), "clocks": clk}
    del x, th, outs
    torch.cuda.empty_cache()
    return r


def run_cfg5(cx, args):
    """configs[4]: ONE 32768x32768 image, G2/H2 M1 + 5-level pyramid, N row bands with halo; the outputs are gathered on
    rank 0 by NCCL, or stored straight into rank 0's planes over NVLink peer memory from inside the fused kernel."""
    torch = cx.torch
    from cvsteer_b200 import bands
    H = W = args.big
    L = 5
    run = bands.BandRun(H, W, L, device=cx.local, world=cx.world, rank=cx.rank)
    run.load_synthetic(seed=5000)
    steps = max(2, min(args.steps, 5))
    px = H * W
    res = {"workload": f"cfg5: one synthetic {W}x{H} image, G2/H2 M1 + 5-level pyramid, {cx.world} row bands with halo",
           "scaling": "strong", "steps": steps, "band_rows_level0": run.band_rows(), "halo_rows_level0": run.halo_rows()}
    ms_c, clk = cx.timed(lambda: run.step("none"), steps, 1)
    res["compute_only_ms"] = round(ms_c, 3)
    res["Mpix_s_compute"] = round(px / 1e6 / (ms_c / 1e3), 1)
    # per level-0 pixel: every level reads its input and writes 3 planes (16 B x 1.332); the stand-alone band-mode pyr_down
    # reads levels 0..3 and writes levels 1..4 once each (4 B x (1.328 + 0.332)); 167 instructions per pixel of every level
    # + 3.75 per pyr_down input pixel
    p03 = sum(0.25 ** l for l in range(4))
    bpp, ipp = 16 * PYR5 + 4 * (p03 + PYR5 - 1), 167 * PYR5 + 3.75 * p03
    res["roofline"] = cx.roofline(px // cx.world, round(bpp, 2), round(ipp, 1), ms_c, "g2_march<M1> + pyr_down per level, band mode")
    res["clocks"] = clk
    if cx.world > 1:
        gb = run.gather_bytes_to_root()
        res["gather_bytes_to_root"] = gb
        for key, mode in (("nccl_gather", "nccl"), ("fused_peer_store", "peer"), ("peer_copy", "copy")):
            try:
                ms, clk2 = cx.timed(lambda: run.step(mode), steps, 1)
                res[key + "_ms"] = round(ms, 3)
                res["Mpix_s_" + key] = round(px / 1e6 / (ms / 1e3), 1)
                res[key + "_root_ingress_GB_s"] = round(gb / 1e9 / (ms / 1e3), 1)
                res[key + "_clocks"] = clk2
            except Exception as ex:   # pragma: no cover - report, do not lose the whole line
                res[key + "_error"] = str(ex)[:300]
        res["collective"] = ("row bands: one gather of the outputs to rank 0 -- ncclSend/ncclRecv grouped per level and overlapped "
                             "with the next level's kernels (nccl_gather), stores from inside the fused kernel into rank 0's planes "
                             "over NVLink peer memory (fused_peer_store), or one copy-engine transfer per level (peer_copy); every "
                             "figure includes the on-stream cross-rank barrier after which rank 0 may read the planes")
        best = min((res[k + "_ms"], k) for k in ("nccl_gather", "fused_peer_store", "peer_copy") if k + "_ms" in res)
        res["best_gather"] = best[1]
        res["best_vs_ingress_bound"] = round(best[0] / (gb / 770e9 * 1e3), 3)
        res["nvlink_peer_GB_s_reference"] = 770.0
    run.close()
    torch.cuda.empty_cache()
    return res


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    from cvsteer_b200.batch import ffma_peak

    assert torch.cuda.is_available(), "bench.py needs a CUDA device: cvsteer_b200 has no CPU fallback"
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=240))
    cx = Ctx(rank, local_rank, world)
    cx.sampler.start()
    try:
        cx.fp32_measured = ffma_peak(0, 20000, local_rank)[0] / 1e12
    except Exception:
        cx.fp32_measured = None

    head = run_headline(cx, args)
    dump = head.pop("dump")
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    e2e = None if args.no_e2e else run_e2e(cx, args, head["state"])
    head.pop("state")
    torch.cuda.empty_cache()

    configs = {}
    want = [c for c in args.configs.split(",") if c]
    for name, fn in (("4k", run_4k_modes), ("cfg3", run_cfg3), ("cfg4", run_cfg4), ("cfg5", run_cfg5)):
        if name not in want:
            continue
        try:
            r = fn(cx, args)
            if name == "4k":
                configs.update(r)
            else:
                configs[name] = r
        except Exception as ex:   # a failing side config must not lose the headline
            configs[name] = {"error": f"{type(ex).__name__}: {ex}"[:400]}
            torch.cuda.empty_cache()

    cx.sampler.stop_flag = True
    cpu = cpu_baseline(args.mode) if (rank == 0 and world == 1 and not args.no_cpu) else None

    if rank == 0:
        line = {"metric": "G2/H2 basis+steer throughput", "value": round(head["value"], 1), "unit": "Mpix/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(head["ms"], 4), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": head["config"],
                "roofline": head["roofline"], "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": head["launches"],
                "clocks": head["clocks"], "configs": configs}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cfg1_line(device=0):
    """configs[0]: host-timed (the call synchronises): 8-bit gray in host memory -> three 8-bit maps in host memory."""
    import ctypes as C

    import numpy as np
    import torch
    from cvsteer_b200 import capi
    root = os.path.dirname(os.path.abspath(__file__))
    fish = np.load(os.path.join(root, "tests", "golden", "fish_fixture.npz"))["fish"]
    rows, cols = fish.shape
    lib = capi.lib()
    h = C.c_void_p()
    capi.check(lib.cvs_g2_create(C.byref(h), device, 4, 0.67))

    def run(batch, outs):
        n = batch.shape[0]
        capi.check(lib.cvs_g2_lines_u8_host(h, batch.data_ptr(), n, rows, cols, cols, rows * cols, 0.0, outs[0].data_ptr(),
                                            outs[1].data_ptr(), outs[2].data_ptr(), cols, rows * cols))

    res = {}
    for n, reps in ((1, 200), (2048, 10)):
        batch = torch.from_numpy(np.repeat(fish[None], n, axis=0)).pin_memory()
        outs = [torch.empty_like(batch).pin_memory() for _ in range(3)]
        for _ in range(3):
            run(batch, outs)
        t0 = time.perf_counter()
        for _ in range(reps):
            run(batch, outs)
        res[n] = (time.perf_counter() - t0) / reps
    from oracle import cvsteer_ref as ref          # CPU leg (cpu_baseline): the oracle, timed beside the GPU path
    import cv2
    cv2.setNumThreads(1)

    def cpu_one():
        _, (g2, h2, e, mag, ph) = ref.g2_full(fish)
        return [ref.normalize_minmax_u8(m) for m in (ref.find_edges(mag, ph), ref.find_dark_lines(mag, ph), ref.find_bright_lines(mag, ph))]
    cpu_one()
    t0 = time.perf_counter()
    for _ in range(20):
        cpu_one()
    t_cpu = (time.perf_counter() - t0) / 20
    lib.cvs_g2_destroy(h)
    px = rows * cols
    return {"config": "cfg1", "what": "cvsteer-run per-file body (gray u8 -> edges / dark lines / bright lines u8) on the bundled %dx%d image" % (cols, rows),
            "n_gpus": 1, "one_file_ms": round(res[1] * 1e3, 4), "one_file_Mpix_s": round(px / 1e6 / res[1], 1),
            "batch_2048_files_ms": round(res[2048] * 1e3, 3), "batch_Mpix_s": round(2048 * px / 1e6 / res[2048], 1),
            "batch_files_per_s": round(2048 / res[2048], 0), "timing": "host wall clock around the synchronous C-ABI call, pinned host buffers",
            "cpu_oracle_one_core_ms": round(t_cpu * 1e3, 3), "cpu_oracle_Mpix_s": round(px / 1e6 / t_cpu, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="M2", choices=list(MODES))
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the e2e leg to the GPU's NUMA node")
    ap.add_argument("--quick", action="store_true", help="skip the sustained run")
    ap.add_argument("--sustain-s", type=float, default=2.0)
    ap.add_argument("--configs", default="4k,cfg3,cfg4,cfg5", help="side configurations to measure (comma list, '' for none)")
    ap.add_argument("--frames-total", type=int, default=256, help="cfg3 / cfg4: frames in total over all GPUs")
    ap.add_argument("--big", type=int, default=32768, help="cfg5: side of the single large image")
    ap.add_argument("--cfg1", action="store_true", help="configs[0] instead: cvsteer-run per-file body on the bundled test image")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of what the last one "
                                                          "computed to DIR/<plane>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.cfg1 or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.cfg1:
        if rank == 0:
            print(json.dumps(cfg1_line(local_rank)), flush=True)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # `python bench.py --gpus N` without torchrun: re-launch under torch.distributed.run
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
