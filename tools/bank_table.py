"""Steering banks against the N single-angle launches a caller runs today, measured in one process with CUDA events.
Writes one JSON object per line to --out:

  - kind "gpu": name, power limit and max SM clock of every visible GPU (nvidia-smi, read in the same run);
  - kind "bank", family "g2": for N in {4, 8, 16} x mask {E, G2T|H2T, STEER5} x {fp32, fp16} planes on 64 x 1080p fp32 frames,
    and for N = 8 on 16 x 4K frames: the bank launch (cvs_g2_steer_bank_dev) and the N launches of steer5@scalar
    (cvs_g2_run_batch_dev_fmt(STEER5, CVS_STEER_SCALAR, theta_k), all five planes, one output set reused);
  - kind "bank", family "g4": for N in {4, 8, 16} x mask {STEER, G4T|H4T} x {fp32, fp16} planes on 64 x 1080p and on
    16 x 4K fp32 frames: the bank launch (cvs_g4_steer_bank_dev) and the N launches of steer@scalar
    (cvs_g4_run_batch_dev_fmt(STEER, CVS_STEER_SCALAR, theta_k), all four planes, one output set reused).
  The two arms alternate round by round after a warm-up of both; rounds x iters, median and spread of the per-round rates.
  Inputs stay resident in HBM and are larger than L2 (530 MB at 1080p, 531 MB at 4K).  Gpix/s counts frame pixels (each bank
  pixel carries N angles), the speed-up is the ratio of the medians, and "of_ceiling" is the bank's rate over its binding
  ceiling: HBM bytes per pixel (4 B in + element size x planes x N out) against MEASURED_PEAKS.json, or the instruction
  estimate below against the nominal fp32 issue rate, whichever is lower.

    python tools/bank_table.py [--out FILE] [--rounds 5] [--iters 10] [--family g2|g4|all]"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from cvsteer_b200 import capi  # noqa: E402
from cvsteer_b200.batch import G2Batch, G4Batch  # noqa: E402
from kernel_table import FP32_NOMINAL, hbm_peak  # noqa: E402

B = capi.bit
# fp32 instructions per pixel (estimates from the source, not counted in SASS): the shared part is the M1 kernel's 167 (basis
# 117 + orientation); per angle the loop adds its control and address arithmetic (~6) plus, per mask, E (6 + 1 store), the
# steering sum (18) with 2 stores, or steering + magnitude / phase (the 199 - 167 + 18 of steer5@scalar) with 5 stores
# G4: the shared part is the basis march of a G4 row, ~323 (DESIGN.md section 9); per angle the loop control and addresses (~6),
# the prescaled steering sum (8 + 17) with 2 stores, or that plus magnitude / phase (~25) with 4 stores
FAMILIES = {
    "g2": dict(cls=G2Batch, instr_shared=167, single_mask=capi.G2_MASK_STEER5, nplanes=capi.G2_NPLANES,
               masks=[("E", B(capi.E), 1, 13), ("G2T|H2T", B(capi.G2T) | B(capi.H2T), 2, 26), ("STEER5", capi.G2_MASK_STEER5, 5, 61)],
               sizes=[((64, 1080, 1920), (4, 8, 16)), ((16, 2160, 3840), (8,))]),
    "g4": dict(cls=G4Batch, instr_shared=323, single_mask=capi.G4_MASK_STEER, nplanes=capi.G4_NPLANES,
               masks=[("G4T|H4T", B(capi.G4T) | B(capi.H4T), 2, 33), ("STEER", capi.G4_MASK_STEER, 4, 60)],
               sizes=[((64, 1080, 1920), (4, 8, 16)), ((16, 2160, 3840), (4, 8, 16))]),
}
FORMATS = [("f32", torch.float32), ("f16", torch.float16)]


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


def spread(v):
    return [min(v), max(v)]


def run_case(fam_name, fam, g, x, n_angles, mask_name, mask, planes, ipa, fmt, dt, a, hbm):
    n, rows, cols = x.shape
    px = n * rows * cols
    thetas = [math.pi * k / n_angles for k in range(n_angles)]
    single_mask, nplanes = fam["single_mask"], fam["nplanes"]
    outs = {p: torch.empty((n_angles, n, rows, cols), dtype=dt, device="cuda") for p in range(nplanes) if mask >> p & 1}
    single = {p: torch.empty((n, rows, cols), dtype=dt, device="cuda") for p in range(nplanes) if single_mask >> p & 1}

    def bank():
        g.steer_bank(x, thetas, mask, outs=outs, out_dtype=dt)

    def launches():
        for th in thetas:
            g.run(x, single_mask, capi.STEER_SCALAR, th, outs=single, out_dtype=dt)

    for _ in range(2):
        bank()
        kname = g.last_launch()["kernel"]
        launches()
        sname = g.last_launch()["kernel"]
    torch.cuda.synchronize()
    rb, rs = [], []
    for _ in range(a.rounds):
        rb.append(px / events_ms(bank, a.iters) / 1e6)
        rs.append(px / events_ms(launches, a.iters) / 1e6)
    esz = 4 if dt == torch.float32 else 2
    bpp = 4 + esz * planes * n_angles
    instr = fam["instr_shared"] + ipa * n_angles
    ceil_hbm, ceil_instr = hbm * 1e9 / bpp / 1e9, FP32_NOMINAL / instr / 1e9
    bound = "hbm" if ceil_hbm <= ceil_instr else "instr"
    mb, ms = statistics.median(rb), statistics.median(rs)
    del outs, single
    torch.cuda.empty_cache()
    return dict(kind="bank", family=fam_name, frames=[n, rows, cols], n_angles=n_angles, mask=mask_name, out=fmt, kernel=kname, single_kernel=sname,
                bank_gpix_s=round(mb, 2), bank_spread=[round(v, 2) for v in spread(rb)], n_launches_gpix_s=round(ms, 2),
                n_launches_spread=[round(v, 2) for v in spread(rs)], speedup=round(mb / ms, 2), bytes_per_px=bpp, instr_per_px_est=instr,
                ceiling_gpix_s=round(min(ceil_hbm, ceil_instr), 1), bound=bound, of_ceiling=round(mb / min(ceil_hbm, ceil_instr), 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_bank_table.jsonl"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--family", choices=["g2", "g4", "all"], default="all")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bank_table measures on a CUDA device"
    hbm = hbm_peak()
    rows_out = [dict(kind="gpu", gpus=gpu_info(), hbm_gbs=hbm, fp32_instr_s=FP32_NOMINAL)]
    for fam_name, fam in FAMILIES.items():
        if a.family not in ("all", fam_name):
            continue
        g = fam["cls"]()
        for shape, ns in fam["sizes"]:
            x = torch.rand(shape, device="cuda") * 255
            for n_angles in ns:
                for mask_name, mask, planes, ipa in fam["masks"]:
                    for fmt, dt in FORMATS:
                        r = run_case(fam_name, fam, g, x, n_angles, mask_name, mask, planes, ipa, fmt, dt, a, hbm)
                        print(json.dumps(r), flush=True)
                        rows_out.append(r)
            del x
        g.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows_out:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
