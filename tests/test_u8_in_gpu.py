"""8-bit input frames with 16-bit output planes and on the host-buffer batch paths.  The fused 8-bit-in / 16-bit-out kernels
and the host-buffer calls write, bit for bit, what the fp32-frame call writes for the same frames widened to float (for
16-bit planes rounded to nearest even); the narrowing fallback writes the fp32 planes of the same 8-bit call, rounded."""
import ctypes as C

import pytest
import torch

from cvsteer_b200 import capi
from cvsteer_b200.batch import G2Batch, G4Batch, pyr_down

pytestmark = pytest.mark.gpu
DTYPES = [torch.float16, torch.bfloat16]
SUFFIX = {torch.float16: "f16", torch.bfloat16: "bf16"}
FMT = {torch.float32: capi.OUT_F32, torch.float16: capi.OUT_F16, torch.bfloat16: capi.OUT_BF16}
SC, MP, DOM = capi.STEER_SCALAR, capi.STEER_MAP, capi.STEER_DOMINANT
G2_CASES = [("M0", capi.G2_MASK_STATE, DOM), ("M1", capi.G2_MASK_ORIENT, DOM), ("M2", capi.G2_MASK_FULL, DOM),
            ("lines", capi.G2_MASK_LINES, DOM), ("M2@scalar", capi.G2_MASK_FULL, SC), ("lines@scalar", capi.G2_MASK_LINES, SC),
            ("steer5@scalar", capi.G2_MASK_STEER5, SC), ("M2@map", capi.G2_MASK_FULL, MP), ("lines@map", capi.G2_MASK_LINES, MP),
            ("steer5@map", capi.G2_MASK_STEER5, MP)]
G4_CASES = [("basis", capi.G4_MASK_BASIS, DOM), ("steer@map", capi.G4_MASK_STEER, MP), ("steer@scalar", capi.G4_MASK_STEER, SC),
            ("steer@theta_d", capi.G4_MASK_STEER, DOM)]
CASES = [(2,) + c for c in G2_CASES] + [(4,) + c for c in G4_CASES]


def same_bits(got, want32, what):
    """got == want32.to(got.dtype) bit for bit, NaN at the same positions."""
    want = want32.to(got.dtype)
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), what
    iview = torch.int16 if got.element_size() == 2 else torch.int32
    bad = (got.view(iview) != want.view(iview)) & ~gn
    assert not bool(bad.any()), (what, int(bad.sum()))


def frames8(seed, n, rows, cols, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    return torch.randint(0, 256, (n, rows, cols), generator=g, device=device, dtype=torch.uint8)


def angles(seed, shape):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(shape, generator=g, device="cuda") * 8.0 - 4.0


def handle(family):
    return G2Batch() if family == 2 else G4Batch()


@pytest.mark.parametrize("shape", [(1080, 1920), (64, 128), (150, 256)])
@pytest.mark.parametrize("case", CASES, ids=[f"g{c[0]}-{c[1]}" for c in CASES])
def test_dense_u8_frames_take_the_fused_kernels(case, shape):
    family, name, mask, src = case
    n = 1 if shape[0] > 1000 else 3
    x8 = frames8(8000 + shape[1], n, *shape)
    g = handle(family)
    kw = dict(steer=src, theta=0.7, theta_map=angles(8100, x8.shape) if src == MP else None)
    r32 = g.run(x8.float(), mask, **kw)
    for dt in DTYPES:
        r = g.run(x8, mask, out_dtype=dt, **kw)
        kern = g.last_launch()["kernel"]
        assert kern.endswith("/tma-u8/imm-taps/" + SUFFIX[dt]) and "+narrow" not in kern, kern
        for k in r32:
            assert r[k].dtype == dt
            same_bits(r[k], r32[k], f"{name} {shape} {dt} {k} ({kern})")


@pytest.mark.parametrize("dt", DTYPES, ids=["f16", "bf16"])
def test_u8_frames_the_fused_kernels_cannot_stage_narrow_with_the_same_bits(dt):
    """Rows TMA cannot stage go through the cooperative 8-bit loader into fp32 scratch and are narrowed: the 16-bit planes are
    the fp32 planes of the same call on the same 8-bit frames (the section 10 contract).  That kernel has no baked taps, so for
    G4 steering at a scalar angle or a map it is not the last-bit twin of the fp32-frame kernel, whose baked taps carry the
    steering factors."""
    pad = frames8(8200, 2, 150, 200)
    for what, x8 in (("pitch of 200 bytes", pad[:, :, :192]), ("130 x 131", frames8(8201, 2, 130, 131))):
        for family, name, mask, src in CASES:
            g = handle(family)
            kw = dict(steer=src, theta=0.7, theta_map=angles(8202, x8.shape) if src == MP else None)
            r32 = g.run(x8, mask, **kw)
            assert g.last_launch()["kernel"].endswith("/ldg-u8"), g.last_launch()["kernel"]
            r = g.run(x8, mask, out_dtype=dt, **kw)
            kern = g.last_launch()["kernel"]
            assert "/ldg-u8" in kern and kern.endswith("+narrow-" + SUFFIX[dt]), kern
            for k in r32:
                same_bits(r[k], r32[k], f"{what} {name} {k}")


def test_pyramid_of_u8_frames():
    x8 = frames8(8300, 2, 540, 960)
    g = G2Batch()
    nl = torch.full((2, 270, 480), float("nan"), device="cuda")
    r = g.run(x8, capi.G2_MASK_FULL, next_level=nl, out_dtype=torch.float16)
    assert g.last_launch()["kernel"] == "g2_march<M2>/tma-u8/imm-taps/f16", g.last_launch()["kernel"]
    assert torch.equal(nl, pyr_down(x8.float()))
    r32 = g.run(x8.float(), capi.G2_MASK_FULL)
    for k in r32:
        same_bits(r[k], r32[k], "level 0 " + k)
    p8 = g.run_pyramid(x8, 3, capi.G2_MASK_FULL, out_dtype=torch.float16)
    p32 = g.run_pyramid(x8.float(), 3, capi.G2_MASK_FULL)
    for l, (a, b) in enumerate(zip(p32, p8)):
        for k in a:
            same_bits(b[k], a[k], f"level {l} {k}")


def _pinned(shape, dtype, pad=0):
    t = torch.empty(shape[:-1] + (shape[-1] + pad,), dtype=dtype, pin_memory=True)
    t.fill_(float("nan") if dtype.is_floating_point else 0)
    return t[..., :shape[-1]] if pad else t


def _host_u8(x8, layout):
    """pinned uint8 host frames holding x8 in one of the layouts the host path copies differently"""
    n, rows, cols = x8.shape
    if layout == "dense":
        h = _pinned((n, rows, cols), torch.uint8)
    elif layout == "padded rows":        # row step and frame step multiples of it: one pitched 3-D copy per chunk
        h = _pinned((n, rows + 3, cols + 40), torch.uint8)[:, :rows, :cols]
    else:                                # frame step not a multiple of the row step: one 2-D copy per frame
        step, fstride = cols + 24, rows * (cols + 24) + 7
        flat = _pinned((n * fstride,), torch.uint8)
        h = flat.as_strided((n, rows, cols), (fstride, step, 1))
    h.copy_(x8.cpu())
    return h


HOST_G2 = [("M0", capi.G2_MASK_STATE), ("M1", capi.G2_MASK_ORIENT), ("M2", capi.G2_MASK_FULL), ("lines", capi.G2_MASK_LINES)]
HOST_G4 = [("basis", capi.G4_MASK_BASIS, None), ("steer@theta_d", capi.G4_MASK_STEER, None), ("steer@scalar", capi.G4_MASK_STEER, 0.7)]
# (layout, n, rows, cols): 1920 columns are dense 128-byte rows; 10 frames leave a short last chunk (chunks of 3)
HOST_GEOMS = [("dense", 10, 270, 1920), ("padded rows", 4, 200, 1920), ("odd frame stride", 3, 130, 392), ("dense", 5, 120, 1000)]


@pytest.mark.parametrize("dt", [torch.float32] + DTYPES, ids=["f32", "f16", "bf16"])
@pytest.mark.parametrize("geom", HOST_GEOMS, ids=[f"{g[0]}-{g[1]}x{g[2]}x{g[3]}" for g in HOST_GEOMS])
def test_host_u8_equals_host_fp32_of_the_widened_frames(geom, dt):
    layout, n, rows, cols = geom
    x8 = frames8(8400 + cols, n, rows, cols)
    xh8 = _host_u8(x8, layout)
    xh32 = _pinned((n, rows, cols), torch.float32)
    xh32.copy_(x8.float().cpu())
    g2, g4 = G2Batch(), G4Batch()
    runs = [(g2, name, mask, {}) for name, mask in HOST_G2] + [(g4, name, mask, {"theta": th}) for name, mask, th in HOST_G4]
    for g, name, mask, kw in runs:
        planes = [p for p in range(len(g._names)) if mask >> p & 1]
        want = {p: _pinned((n, rows, cols), dt) for p in planes}
        got = {p: _pinned((n, rows, cols), dt, pad=8) for p in planes}
        g.run_host(xh32, mask, want, **kw)
        g.run_host(xh8, mask, got, **kw)
        for p in planes:
            same_bits(got[p], want[p], f"{layout} {name} plane {p}")


@pytest.mark.parametrize("dt", [torch.float32] + DTYPES, ids=["f32", "f16", "bf16"])
def test_multi_gpu_host_u8_equals_the_widened_frames(dt):
    n, rows, cols = 7, 270, 1920
    ndev = torch.cuda.device_count()
    devices = [0, 0] if ndev == 1 else list(range(ndev))
    dev_arr = (C.c_int * len(devices))(*devices)
    x8 = frames8(8500, n, rows, cols)
    xh8 = _host_u8(x8, "dense")
    xh32 = _pinned((n, rows, cols), torch.float32)
    xh32.copy_(x8.float().cpu())
    es = torch.empty((), dtype=dt).element_size()
    planes = [p for p in range(capi.G2_NPLANES) if capi.G2_MASK_FULL >> p & 1]
    lib = capi.lib()
    res = []
    for fn, x, in_es in ((lib.cvs_g2_run_batch_host_multi_fmt, xh32, 4), (lib.cvs_g2_run_batch_host_multi_u8, xh8, 1)):
        outs = {p: _pinned((n, rows, cols), dt) for p in planes}
        arr = (C.c_void_p * capi.G2_NPLANES)()
        for p, t in outs.items():
            arr[p] = t.data_ptr()
        capi.check(fn(len(devices), dev_arr, 4, 0.67, C.c_void_p(x.data_ptr()), n, rows, cols, cols * in_es, rows * cols * in_es,
                      capi.G2_MASK_FULL, arr, cols * es, rows * cols * es, FMT[dt]))
        res.append(outs)
    for p in planes:
        same_bits(res[1][p], res[0][p], f"multi plane {p}")


def test_run_host_rejects_frames_it_cannot_read():
    g2, g4 = G2Batch(), G4Batch()
    outs = {capi.E: _pinned((2, 32, 64), torch.float32)}
    outs4 = {capi.MAG4: _pinned((2, 32, 64), torch.float32)}
    lib = capi.lib()
    before = lib.cvs_launch_count()
    bad = [torch.zeros((2, 32, 64), dtype=torch.float64), torch.zeros((2, 32, 64), dtype=torch.int16),
           torch.zeros((2, 32, 64), dtype=torch.uint8, device="cuda"), torch.zeros((2, 32, 64), device="cuda"),
           torch.zeros((2, 64, 32), dtype=torch.uint8).transpose(1, 2)]
    for x in bad:
        with pytest.raises(capi.CvsError) as e:
            g2.run_host(x, capi.bit(capi.E), outs)
        assert e.value.code == capi.ERR_INVALID_ARG
        with pytest.raises(capi.CvsError):
            g4.run_host(x, capi.bit(capi.MAG4), outs4)
    assert lib.cvs_launch_count() == before
