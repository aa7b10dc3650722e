"""G4/H4 steering banks on the device: every plane bit for bit (NaN positions included) what the single-angle call the
contract names writes on the same handle -- cvs_g4_run_batch_dev_fmt(CVS_G4_MASK_STEER, CVS_STEER_SCALAR, thetas[k]) per
angle, on the frames as fp32 (8-bit frames widened to float) -- for the fused kernel (one launch) and the fallback."""
import ctypes as C
import math

import pytest
import torch

from cvsteer_b200 import capi
from cvsteer_b200.batch import Band, G2Batch, G4Batch, _batch_struct, pyr_down

pytestmark = pytest.mark.gpu

B = capi.bit
MASKS = [capi.G4_MASK_STEER, B(capi.G4T) | B(capi.H4T), B(capi.MAG4) | B(capi.PHASE4), B(capi.H4T)]
# 0, +-pi/2, +-pi, +-7 rad and a repeated angle come first, so every bank of 8 or more angles has them all
ANGLES = [0.0, math.pi / 2, -math.pi / 2, math.pi, -math.pi, 7.0, -7.0, 0.3, 0.3, 1.1, -2.5, 2.9, -0.01, 3.3, -4.4, 0.77]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
FMT = {torch.float32: "", torch.float16: "/f16", torch.bfloat16: "/bf16"}


def _bits(t):
    return t.view({4: torch.int32, 2: torch.int16}[t.element_size()])


def _same(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape)
    eq = _bits(a) == _bits(b)
    assert bool(eq.all()), (what, int((~eq).sum()))


def _frames(n, rows, cols, u8, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand((n, rows, cols), generator=g, device="cuda") * 255
    # a flat patch: zero basis response there, so the phase of a vanishing response
    x[:, : rows // 8, : cols // 8] = 17.0
    return x.to(torch.uint8) if u8 else x


class Ref:
    """The single-angle calls of the contract, on the frames as fp32, cached per angle."""

    def __init__(self, g, x, dtype, band=None):
        self.g, self.x, self.dtype, self.band, self.cache = g, x.float() if x.dtype == torch.uint8 else x, dtype, band, {}

    def angle(self, th):
        if th not in self.cache:
            self.cache[th] = self.g.run(self.x, capi.G4_MASK_STEER, capi.STEER_SCALAR, th, out_dtype=self.dtype, band=self.band)
        return self.cache[th]

    def check(self, got, thetas, mask, what):
        for p in range(capi.G4_NPLANES):
            if mask >> p & 1:
                name = capi.G4_PLANE_NAMES[p]
                for k, th in enumerate(thetas):
                    _same(got[name][k], self.angle(th)[name], (what, name, k, th))


def _bank(g, x, thetas, mask, **kw):
    lib = capi.lib()
    before = lib.cvs_launch_count()
    r = g.steer_bank(x, thetas, mask, **kw)
    torch.cuda.synchronize()
    return r, lib.cvs_launch_count() - before, g.last_launch()["kernel"]


@pytest.mark.parametrize("shape", [(2, 1080, 1920), (3, 64, 128)])
@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("dtype", DTYPES)
def test_fused_g4_bank_matches_single_angle_calls(shape, u8, dtype):
    g = G4Batch()
    x = _frames(*shape, u8)
    ref = Ref(g, x, dtype)
    want = f"g4_bank/{'tma-u8' if u8 else 'tma'}/imm-taps{FMT[dtype]}"
    for n_angles in (1, 3, 8, 16):
        thetas = ANGLES[:n_angles]
        for mask in MASKS:
            got, launches, kernel = _bank(g, x, thetas, mask, out_dtype=dtype)
            assert kernel == want and launches == 1, (kernel, launches)
            assert sorted(got) == sorted(capi.G4_PLANE_NAMES[p] for p in range(capi.G4_NPLANES) if mask >> p & 1)
            for t in got.values():
                assert tuple(t.shape) == (n_angles,) + shape
            ref.check(got, thetas, mask, (n_angles, hex(mask)))
    # the single-angle kernel the fused bank replaces is steer@scalar with baked taps
    g.run(ref.x, capi.G4_MASK_STEER, capi.STEER_SCALAR, 0.3, out_dtype=dtype)
    assert g.last_launch()["kernel"].startswith("g4_march<steer@scalar>/tma/imm-taps")


def test_u8_frames_follow_the_widened_frames_call():
    # With fp32 planes the single-angle call on 8-bit frames runs the constant-bank /tma-u8 kernel, whose taps are not
    # prescaled: its last bits differ from the call on the widened frames.  The bank gives the widened-frames bits.
    g = G4Batch()
    x = _frames(2, 1080, 1920, True, seed=4)
    thetas = [0.3, -1.2, 2.5]
    got, launches, kernel = _bank(g, x, thetas, capi.G4_MASK_STEER)
    assert kernel == "g4_bank/tma-u8/imm-taps" and launches == 1
    Ref(g, x, torch.float32).check(got, thetas, capi.G4_MASK_STEER, "u8 = widened")
    direct = g.run(x, capi.G4_MASK_STEER, capi.STEER_SCALAR, thetas[0])
    assert g.last_launch()["kernel"] == "g4_march<steer@scalar>/tma-u8"
    assert not bool((_bits(direct["g4"]) == _bits(got["g4"][0])).all()), "the 8-bit single-angle kernel now prescales: revisit the contract"


def _fallback_case(g, x, dtype, thetas=ANGLES[:5], mask=capi.G4_MASK_STEER, **kw):
    got, launches, kernel = _bank(g, x, thetas, mask, out_dtype=dtype, **kw)
    assert kernel.startswith("bank-fallback:"), kernel
    assert launches >= len(thetas)  # one launch per angle (16-bit planes may add a narrowing launch, 8-bit frames a widening one)
    Ref(g, x, dtype).check(got, thetas, mask, kernel)
    return kernel


@pytest.mark.parametrize("dtype", DTYPES)
def test_g4_fallback_forms(dtype):
    g = G4Batch()
    # cooperative loader (130 x 131 frames: rows of 524 bytes), fp32 and 8-bit (widened to the same dense fp32 layout)
    k = _fallback_case(g, _frames(2, 130, 131, False), dtype)
    assert "/ldg" in k and "u8" not in k
    k = _fallback_case(g, _frames(2, 130, 131, True), dtype, mask=B(capi.G4T) | B(capi.PHASE4))
    assert "/ldg" in k and "u8" not in k
    # a 200-byte input pitch
    padded = _frames(2, 96, 50, False)[:, :, :48]
    assert padded.stride(1) * 4 == 200
    _fallback_case(g, padded, dtype)
    # non-default spacing (constant-bank taps), width 5 (the generic path)
    _fallback_case(G4Batch(spacing=0.4), _frames(2, 96, 128, False), dtype, mask=B(capi.H4T) | B(capi.MAG4))
    _fallback_case(G4Batch(width=5), _frames(2, 96, 128, False), dtype, mask=B(capi.G4T))
    _fallback_case(G4Batch(width=5), _frames(2, 96, 128, True), dtype, mask=B(capi.PHASE4))


def test_g4_fallback_u8_frames_fp32_planes():
    # 8-bit frames with fp32 planes where the fused bank does not apply: the fallback widens them first, so it gives the
    # widened-frames bits too (and not those of the 8-bit single-angle kernels)
    x = _frames(2, 130, 131, True, seed=5)
    for g in (G4Batch(), G4Batch(spacing=0.45)):
        k = _fallback_case(g, x, torch.float32, thetas=ANGLES[:8])
        assert "u8" not in k


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_g4_layouts(dtype):
    g = G4Batch()
    n, rows, cols, N = 3, 200, 256, 6
    x = _frames(n, rows, cols, False, seed=1)
    thetas = ANGLES[2:2 + N]
    mask = capi.G4_MASK_STEER
    ref = Ref(g, x, dtype)
    planes = [p for p in range(capi.G4_NPLANES) if mask >> p & 1]
    # frame-major: [n, N, rows, cols] storage seen as [N, n, rows, cols]
    outs = {p: torch.empty((n, N, rows, cols), dtype=dtype, device="cuda").transpose(0, 1) for p in planes}
    got, launches, kernel = _bank(g, x, thetas, mask, outs=outs, out_dtype=dtype)
    assert kernel.startswith("g4_bank/") and launches == 1
    ref.check(got, thetas, mask, "frame-major")
    # padded pitches (rows of cols + 24 elements)
    outs = {p: torch.empty((N, n, rows, cols + 24), dtype=dtype, device="cuda")[..., :cols] for p in planes}
    got, launches, kernel = _bank(g, x, thetas, mask, outs=outs, out_dtype=dtype)
    assert kernel.startswith("g4_bank/") and launches == 1
    ref.check(got, thetas, mask, "padded")


def test_g4_batch_fields():
    g = G4Batch()
    n, rows, cols = 2, 540, 960
    x = _frames(n, rows, cols, False, seed=2)
    thetas = ANGLES[:8]
    nxt = torch.empty((n, (rows + 1) // 2, (cols + 1) // 2), device="cuda")
    _, launches, kernel = _bank(g, x, thetas, capi.G4_MASK_STEER, next_level=nxt)
    assert kernel.startswith("g4_bank/") and launches == 1
    _same(nxt, pyr_down(x), "next_level")
    for dtype in (torch.float32, torch.bfloat16):
        whole = g.steer_bank(x, thetas, capi.G4_MASK_STEER, out_dtype=dtype)
        for r0, r1 in ((0, 100), (130, 397), (400, rows)):
            part, launches, kernel = _bank(g, x, thetas, capi.G4_MASK_STEER, band=Band(rows, 0, r0, r1), out_dtype=dtype)
            assert kernel.startswith("g4_bank/") and launches == 1
            for name, t in part.items():
                _same(t, whole[name][..., r0:r1, :], ("band", name, r0, r1))
    # the fallback honours them as well (width 5: the generic path, pyr_down on its own)
    g5 = G4Batch(width=5)
    nxt5 = torch.empty_like(nxt)
    _, _, kernel = _bank(g5, x, thetas[:3], capi.G4_MASK_STEER, next_level=nxt5)
    assert kernel.startswith("bank-fallback:")
    _same(nxt5, pyr_down(x), "fallback next_level")


def test_bank_calls_take_their_own_family_only():
    lib = capi.lib()
    g2, g4 = G2Batch(), G4Batch()
    x = _frames(1, 64, 128, False)
    out = torch.empty((1, 1, 64, 128), device="cuda")
    b = _batch_struct(x, 128 * 4, 64 * 128 * 4, None)
    th = (C.c_float * 1)(0.5)
    for fn, h, p in ((lib.cvs_g4_steer_bank_dev, g2._h, capi.G4T), (lib.cvs_g2_steer_bank_dev, g4._h, capi.G2T)):
        arr = (C.c_void_p * capi.G2_NPLANES)()
        arr[p] = out.data_ptr()
        before = lib.cvs_launch_count()
        assert fn(h, C.byref(b), th, 1, B(p), arr, 0, None, capi.OUT_F32) == capi.ERR_INVALID_ARG
        assert b"handle" in lib.cvs_last_error() and lib.cvs_launch_count() == before


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("dtype", DTYPES)
def test_g4_host_call_matches_device_bank(u8, dtype):
    g = G4Batch()
    n, rows, cols = 7, 64, 128  # 7 frames: chunks of 2, 2, 2 and a short last one of 1
    thetas = ANGLES[3:8]
    mask = capi.G4_MASK_STEER
    xd = _frames(n, rows, cols, u8, seed=3)
    xh = xd.cpu().pin_memory()
    want = g.steer_bank(xd, thetas, mask, out_dtype=dtype)
    assert g.last_launch()["kernel"].startswith("g4_bank/")
    outs = {p: torch.full((len(thetas), n, rows, cols), float("nan"), dtype=dtype).pin_memory()
            for p in range(capi.G4_NPLANES) if mask >> p & 1}
    g.steer_bank_host(xh, thetas, mask, outs)
    for p, t in outs.items():
        _same(t, want[capi.G4_PLANE_NAMES[p]].cpu(), ("host", p))
    # frame-major host planes with padded rows
    outs2 = {p: torch.zeros((n, len(thetas), rows, cols + 8), dtype=dtype).pin_memory().transpose(0, 1)[..., :cols] for p in outs}
    g.steer_bank_host(xh, thetas, mask, outs2)
    for p, t in outs2.items():
        _same(t.contiguous(), want[capi.G4_PLANE_NAMES[p]].cpu(), ("host frame-major", p))
