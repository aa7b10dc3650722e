"""16-bit output planes (out_dtype float16 / bfloat16, the *_fmt entry points): every plane equals, bit for bit, the fp32 plane
of the same call rounded to nearest even (torch's .to()), whichever kernel wrote it -- the fused 16-bit kernels or the
fp32-kernel-into-scratch + narrowing fallback."""
import ctypes as C

import numpy as np
import pytest
import torch

from cvsteer_b200 import capi
from cvsteer_b200.batch import Band, G2Batch, G4Batch

pytestmark = pytest.mark.gpu
DTYPES = [torch.float16, torch.bfloat16]
SUFFIX = {torch.float16: "f16", torch.bfloat16: "bf16"}
FMT = {torch.float16: capi.OUT_F16, torch.bfloat16: capi.OUT_BF16}
SC, MP, DOM = capi.STEER_SCALAR, capi.STEER_MAP, capi.STEER_DOMINANT
G2_CASES = [("M0", capi.G2_MASK_STATE, DOM), ("M1", capi.G2_MASK_ORIENT, DOM), ("M2", capi.G2_MASK_FULL, DOM),
            ("lines", capi.G2_MASK_LINES, DOM), ("M2@scalar", capi.G2_MASK_FULL, SC), ("lines@scalar", capi.G2_MASK_LINES, SC),
            ("steer5@scalar", capi.G2_MASK_STEER5, SC), ("M2@map", capi.G2_MASK_FULL, MP), ("lines@map", capi.G2_MASK_LINES, MP),
            ("steer5@map", capi.G2_MASK_STEER5, MP)]
G4_CASES = [("basis", capi.G4_MASK_BASIS, DOM), ("steer@map", capi.G4_MASK_STEER, MP), ("steer@scalar", capi.G4_MASK_STEER, SC),
            ("steer@theta_d", capi.G4_MASK_STEER, DOM)]
CASES = [(2,) + c for c in G2_CASES] + [(4,) + c for c in G4_CASES]


def same_bits(got, want32, what):
    """got (16-bit) == want32.to(got.dtype) bit for bit, NaN at the same positions."""
    want = want32.to(got.dtype)
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), what
    bad = (got.view(torch.int16) != want.view(torch.int16)) & ~gn
    assert not bool(bad.any()), (what, int(bad.sum()))


def frames(seed, n, rows, cols):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand((n, rows, cols), generator=g, device="cuda") * 255.0


def angles(seed, shape):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(shape, generator=g, device="cuda") * 8.0 - 4.0


def handle(family, **kw):
    return G2Batch(**kw) if family == 2 else G4Batch(**kw)


def run_both(g, x, mask, src, tm=None, **kw):
    """fp32 planes, then {dtype: (16-bit planes, kernel name)}"""
    args = dict(steer=src, theta=0.7, theta_map=tm if src == MP else None, **kw)
    r32 = g.run(x, mask, **args)
    out = {}
    for dt in DTYPES:
        r = g.run(x, mask, out_dtype=dt, **args)
        out[dt] = (r, g.last_launch()["kernel"])
    return r32, out


@pytest.mark.parametrize("shape", [(1080, 1920), (130, 131), (64, 128), (37, 5)])
@pytest.mark.parametrize("case", CASES, ids=[f"g{c[0]}-{c[1]}" for c in CASES])
def test_every_named_mask_and_source_narrows_bit_exactly(case, shape):
    family, name, mask, src = case
    n = 1 if shape[0] > 1000 else 2
    x = frames(7000 + shape[1], n, *shape)
    g = handle(family)
    r32, res = run_both(g, x, mask, src, angles(7100, x.shape))
    for dt, (r, kern) in res.items():
        # dense rows of a multiple of 4 columns: TMA tile and 4-byte pair stores, i.e. the fused 16-bit kernel
        if shape[1] % 4 == 0:
            assert kern.endswith("/" + SUFFIX[dt]) and "+narrow" not in kern, kern
        else:
            assert kern.endswith("+narrow-" + SUFFIX[dt]), kern
        for k in r32:
            assert r[k].dtype == dt
            same_bits(r[k], r32[k], f"{name} {shape} {dt} {k} ({kern})")


@pytest.mark.parametrize("shape", [(1080, 1920), (2160, 3840)])
def test_dense_frames_take_the_fused_16_bit_kernels(shape):
    x = frames(7200, 1, *shape)
    tm = angles(7201, x.shape)
    for family, name, mask, src in CASES:
        g = handle(family)
        r32, res = run_both(g, x, mask, src, tm)
        for dt, (r, kern) in res.items():
            assert kern.endswith("/tma/imm-taps/2px/" + SUFFIX[dt]) or kern.endswith("/tma/imm-taps/" + SUFFIX[dt]), kern
            for k in r32:
                same_bits(r[k], r32[k], f"{name} {shape} {k}")


def _run_fmt(g, x, mask, dt, pitch_elems, src=DOM, theta_map=None, theta_pitch_elems=None):
    """16-bit planes through cvs_*_run_batch_dev_fmt with a row pitch of pitch_elems elements; returns views [n, rows, cols]."""
    n, rows, cols = x.shape
    planes = [p for p in range(len(g._names)) if mask >> p & 1]
    bufs = {p: torch.full((n, rows, pitch_elems), float("nan"), dtype=dt, device="cuda") for p in planes}
    arr = (C.c_void_p * len(g._names))()
    for p in planes:
        arr[p] = bufs[p].data_ptr()
    b = capi.Batch()
    b.in_, b.in_is_u8, b.n, b.rows, b.cols = x.data_ptr(), 0, n, rows, cols
    b.in_pitch, b.in_frame_stride = x.stride(1) * 4, x.stride(0) * 4
    b.out_pitch, b.out_frame_stride = pitch_elems * 2, pitch_elems * 2 * rows
    tm = C.c_void_p(theta_map.data_ptr()) if theta_map is not None else None
    fn = getattr(g._lib, f"cvs_{g._prefix}_run_batch_dev_fmt")
    capi.check(fn(g._h, C.byref(b), mask, src, 0.7, tm, arr, C.c_void_p(torch.cuda.current_stream().cuda_stream), FMT[dt]))
    return {g._names[p]: bufs[p][:, :, :cols] for p in planes}, g.last_launch()["kernel"]


@pytest.mark.parametrize("dt", DTYPES, ids=["f16", "bf16"])
def test_fallback_geometries_give_the_same_bits(dt):
    x = frames(7300, 2, 300, 392)
    g = G2Batch()
    full = capi.G2_MASK_FULL
    r32 = g.run(x, full)
    # unaligned pitch (2-byte but not 4-byte aligned rows): the two-pixel kernel cannot store pairs
    r, kern = _run_fmt(g, x, full, dt, 393)
    assert kern.endswith("+narrow-" + SUFFIX[dt]), kern
    for k in r32:
        same_bits(r[k], r32[k], "unaligned pitch " + k)
    # 8-bit input
    xu = x.to(torch.uint8)
    a, b = g.run(xu, full), g.run(xu, full, out_dtype=dt)
    assert g.last_launch()["kernel"].endswith("+narrow-" + SUFFIX[dt])
    for k in a:
        same_bits(b[k], a[k], "u8 " + k)
    # width-3 taps (generic path)
    g3 = G2Batch(width=3)
    a, b = g3.run(x, full), g3.run(x, full, out_dtype=dt)
    assert g3.last_launch()["kernel"].startswith("generic_w3") and g3.last_launch()["kernel"].endswith("+narrow-" + SUFFIX[dt])
    for k in a:
        same_bits(b[k], a[k], "width 3 " + k)
    # run-time mask, with the fused next pyramid level (stays fp32, same bits as the fp32 call's)
    dyn = full | capi.bit(capi.G2A)
    nl32 = torch.empty((2, 150, 196), device="cuda")
    nl16 = torch.full_like(nl32, float("nan"))
    a, b = g.run(x, dyn, next_level=nl32), g.run(x, dyn, next_level=nl16, out_dtype=dt)
    assert g.last_launch()["kernel"] == "g2_march<dyn>/tma+narrow-" + SUFFIX[dt], g.last_launch()["kernel"]
    assert torch.equal(nl16, nl32)
    for k in a:
        same_bits(b[k], a[k], "dyn " + k)
    # band mode: rows [100, 200) of frame 0 from a buffer holding rows [90, 210); equals the whole-frame slice too
    band = Band(full_rows=300, y_origin=90, row_begin=100, row_end=200)
    a, b = g.run(x[:1, 90:210], full, band=band), g.run(x[:1, 90:210], full, band=band, out_dtype=dt)
    whole = g.run(x[:1], full, out_dtype=dt)
    for k in a:
        same_bits(b[k], a[k], "band " + k)
        assert torch.equal(b[k].view(torch.int16), whole[k][:, 100:200].view(torch.int16)), "band vs whole " + k
    # CVS_STEER_MAP with a strided layout: out pitch 400 elements, the fp32 angle map in the same element layout
    tm = angles(7301, (2, 300, 400))
    for mask in (capi.G2_MASK_STEER5, capi.G2_MASK_LINES):
        a = g.run(x, mask, steer=MP, theta_map=tm[:, :, :392].contiguous())
        b, kern = _run_fmt(g, x, mask, dt, 400, src=MP, theta_map=tm)
        for k in a:
            same_bits(b[k], a[k], f"strided map {mask:#x} {k} ({kern})")


@pytest.mark.parametrize("dt", DTYPES, ids=["f16", "bf16"])
def test_pyramid_levels_narrow_and_next_level_stays_fp32(dt):
    x = frames(7400, 2, 540, 960)
    g = G2Batch()
    p32 = g.run_pyramid(x, 3, capi.G2_MASK_FULL)
    p16 = g.run_pyramid(x, 3, capi.G2_MASK_FULL, out_dtype=dt)
    for l, (a, b) in enumerate(zip(p32, p16)):
        for k in a:
            same_bits(b[k], a[k], f"level {l} {k}")
    nl32 = torch.empty((2, 270, 480), device="cuda")
    nl16 = torch.full_like(nl32, float("nan"))
    g.run(x, capi.G2_MASK_FULL, next_level=nl32)
    g.run(x, capi.G2_MASK_FULL, next_level=nl16, out_dtype=dt)
    assert g.last_launch()["kernel"].endswith("/" + SUFFIX[dt])
    assert torch.equal(nl16, nl32)


def test_fp16_overflow_is_inf_where_narrowing_puts_it():
    x = frames(7500, 1, 1080, 1920)
    g = G2Batch()
    r32 = g.run(x, capi.G2_MASK_FULL)
    r16 = g.run(x, capi.G2_MASK_FULL, out_dtype=torch.float16)
    rbf = g.run(x, capi.G2_MASK_FULL, out_dtype=torch.bfloat16)
    for k in ("strength", "e"):
        assert bool(torch.isinf(r16[k]).any()), k     # the quadratic planes of [0,255) frames pass 65504
        assert torch.equal(torch.isinf(r16[k]), r32[k].abs() >= 65520.0), k
        same_bits(r16[k], r32[k], "f16 " + k)
        assert not bool(torch.isinf(rbf[k]).any()), k


def _pinned(shape, dtype, pad=0):
    t = torch.empty(shape[:-1] + (shape[-1] + pad,), dtype=dtype, pin_memory=True)
    t.fill_(float("nan"))
    return t[..., :shape[-1]] if pad else t


@pytest.mark.parametrize("dt", DTYPES, ids=["f16", "bf16"])
def test_host_paths_equal_the_device_path(dt):
    n, rows, cols = 5, 270, 1920
    xd = frames(7600, n, rows, cols)
    xh = _pinned((n, rows, cols), torch.float32)
    xh.copy_(xd.cpu())
    g2, g4 = G2Batch(), G4Batch()
    for pad in (0, 64):   # dense planes (one linear copy per plane and chunk) and strided host rows
        want = g2.run(xd, capi.G2_MASK_FULL, out_dtype=dt)
        outs = {p: _pinned((n, rows, cols), dt, pad) for p in range(capi.G2_NPLANES) if capi.G2_MASK_FULL >> p & 1}
        g2.run_host(xh, capi.G2_MASK_FULL, outs)
        for p, t in outs.items():
            assert torch.equal(t.view(torch.int16), want[capi.G2_PLANE_NAMES[p]].cpu().view(torch.int16)), (pad, p)
        for theta in (None, 0.7):
            src = DOM if theta is None else SC
            want = g4.run(xd, capi.G4_MASK_STEER, steer=src, theta=theta or 0.0, out_dtype=dt)
            outs = {p: _pinned((n, rows, cols), dt, pad) for p in range(capi.G4_NPLANES) if capi.G4_MASK_STEER >> p & 1}
            g4.run_host(xh, capi.G4_MASK_STEER, outs, theta=theta)
            for p, t in outs.items():
                assert torch.equal(t.view(torch.int16), want[capi.G4_PLANE_NAMES[p]].cpu().view(torch.int16)), (pad, theta, p)
    # frame sharding over every visible GPU
    ndev = torch.cuda.device_count()
    outs = {p: _pinned((n, rows, cols), dt) for p in range(capi.G2_NPLANES) if capi.G2_MASK_FULL >> p & 1}
    arr = (C.c_void_p * capi.G2_NPLANES)()
    for p, t in outs.items():
        arr[p] = t.data_ptr()
    capi.check(capi.lib().cvs_g2_run_batch_host_multi_fmt(ndev, None, 4, 0.67, C.c_void_p(xh.data_ptr()), n, rows, cols, cols * 4,
                                                          rows * cols * 4, capi.G2_MASK_FULL, arr, cols * 2, rows * cols * 2, FMT[dt]))
    want = g2.run(xd, capi.G2_MASK_FULL, out_dtype=dt)
    for p, t in outs.items():
        assert torch.equal(t.view(torch.int16), want[capi.G2_PLANE_NAMES[p]].cpu().view(torch.int16)), ("multi", p)


def test_f32_through_the_fmt_calls_is_the_fp32_call():
    n, rows, cols = 3, 200, 392
    xd = frames(7700, n, rows, cols)
    g = G2Batch()
    lib = capi.lib()
    want = g.run(xd, capi.G2_MASK_FULL)
    name = g.last_launch()["kernel"]
    outs = {p: torch.full((n, rows, cols), float("nan"), device="cuda") for p in range(capi.G2_NPLANES) if capi.G2_MASK_FULL >> p & 1}
    arr = (C.c_void_p * capi.G2_NPLANES)()
    for p, t in outs.items():
        arr[p] = t.data_ptr()
    b = capi.Batch()
    b.in_, b.n, b.rows, b.cols = xd.data_ptr(), n, rows, cols
    b.in_pitch, b.in_frame_stride, b.out_pitch, b.out_frame_stride = cols * 4, rows * cols * 4, cols * 4, rows * cols * 4
    capi.check(lib.cvs_g2_run_batch_dev_fmt(g._h, C.byref(b), capi.G2_MASK_FULL, DOM, 0.0, None, arr,
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream), capi.OUT_F32))
    torch.cuda.synchronize()
    assert g.last_launch()["kernel"] == name
    for p, t in outs.items():
        assert torch.equal(t, want[capi.G2_PLANE_NAMES[p]]), p
    # host and multi-GPU host calls
    xh = _pinned((n, rows, cols), torch.float32)
    xh.copy_(xd.cpu())
    for multi in (False, True):
        old = {p: _pinned((n, rows, cols), torch.float32) for p in outs}
        new = {p: _pinned((n, rows, cols), torch.float32) for p in outs}
        for o, fmt in ((old, None), (new, capi.OUT_F32)):
            arr = (C.c_void_p * capi.G2_NPLANES)()
            for p, t in o.items():
                arr[p] = t.data_ptr()
            common = (C.c_void_p(xh.data_ptr()), n, rows, cols, cols * 4, rows * cols * 4, capi.G2_MASK_FULL, arr, cols * 4, rows * cols * 4)
            if multi:
                pre = (torch.cuda.device_count(), None, 4, 0.67)
                rc = lib.cvs_g2_run_batch_host_multi(*pre, *common) if fmt is None else lib.cvs_g2_run_batch_host_multi_fmt(*pre, *common, fmt)
            else:
                rc = lib.cvs_g2_run_batch_host(g._h, *common) if fmt is None else lib.cvs_g2_run_batch_host_fmt(g._h, *common, fmt)
            capi.check(rc)
        for p in outs:
            assert torch.equal(old[p], new[p]) and torch.equal(old[p], want[capi.G2_PLANE_NAMES[p]].cpu()), (multi, p)
