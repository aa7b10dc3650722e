"""Steering banks on the device: every plane bit for bit (NaN positions included) what the single-angle calls the contract
names write on the same handle and batch -- cvs_g2_run_batch_dev_fmt(STEER5, CVS_STEER_SCALAR, thetas[k]) per angle and
CVS_G2_MASK_ORIENT at theta_d for theta / strength -- for the fused kernel (one launch) and the fallback."""
import math

import numpy as np
import pytest
import torch

from cvsteer_b200 import capi
from cvsteer_b200.batch import Band, G2Batch, pyr_down

pytestmark = pytest.mark.gpu

B = capi.bit
MASKS = [capi.G2_MASK_STEER5, B(capi.E), B(capi.G2T) | B(capi.H2T), B(capi.MAG) | B(capi.PHASE), capi.G2_BANK_PLANES]
# 0, +-pi/2, +-pi, +-7 rad and a repeated angle come first, so every bank of 8 or more angles has them all
ANGLES = [0.0, math.pi / 2, -math.pi / 2, math.pi, -math.pi, 7.0, -7.0, 0.3, 0.3, 1.1, -2.5, 2.9, -0.01, 3.3, -4.4, 0.77]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
ONCE = (capi.THETA, capi.STRENGTH)


def _bits(t):
    return t.view({4: torch.int32, 2: torch.int16}[t.element_size()])


def _same(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape)
    eq = _bits(a) == _bits(b)
    assert bool(eq.all()), (what, int((~eq).sum()))


def _frames(n, rows, cols, u8, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand((n, rows, cols), generator=g, device="cuda") * 255
    # a flat patch: zero basis response there, so strength 0 and the angle / phase of a vanishing response
    x[:, : rows // 8, : cols // 8] = 17.0
    return x.to(torch.uint8) if u8 else x


class Ref:
    """The single-angle calls of the contract, cached per angle."""

    def __init__(self, g, x, dtype, band=None):
        self.g, self.x, self.dtype, self.band, self.cache = g, x, dtype, band, {}

    def angle(self, th):
        if th not in self.cache:
            self.cache[th] = self.g.run(self.x, capi.G2_MASK_STEER5, capi.STEER_SCALAR, th, out_dtype=self.dtype, band=self.band)
        return self.cache[th]

    def orient(self):
        if "orient" not in self.cache:
            self.cache["orient"] = self.g.run(self.x, capi.G2_MASK_ORIENT, out_dtype=self.dtype, band=self.band)
        return self.cache["orient"]

    def check(self, got, thetas, mask, what):
        for p in range(capi.G2_NPLANES):
            if not mask >> p & 1:
                continue
            name = capi.G2_PLANE_NAMES[p]
            if p in ONCE:
                _same(got[name], self.orient()[name], (what, name))
            else:
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
def test_fused_bank_matches_single_angle_calls(shape, u8, dtype):
    g = G2Batch()
    x = _frames(*shape, u8)
    ref = Ref(g, x, dtype)
    fmt = {torch.float32: "", torch.float16: "/f16", torch.bfloat16: "/bf16"}[dtype]
    want = f"g2_bank/{'tma-u8' if u8 else 'tma'}/imm-taps{fmt}"
    for n_angles in (1, 3, 8, 16):
        thetas = ANGLES[:n_angles]
        for mask in MASKS:
            got, launches, kernel = _bank(g, x, thetas, mask, out_dtype=dtype)
            assert kernel.startswith("g2_bank/") and kernel == want, kernel
            assert launches == 1
            for p in range(capi.G2_NPLANES):
                if mask >> p & 1:
                    t = got[capi.G2_PLANE_NAMES[p]]
                    assert tuple(t.shape) == ((shape if p in ONCE else (n_angles,) + shape)), (p, t.shape)
            ref.check(got, thetas, mask, (n_angles, hex(mask)))


def _fallback_case(g, x, dtype, thetas=ANGLES[:5], mask=capi.G2_BANK_PLANES, **kw):
    got, launches, kernel = _bank(g, x, thetas, mask, out_dtype=dtype, **kw)
    assert kernel.startswith("bank-fallback:"), kernel
    # at least one launch per angle, and one ORIENT launch when theta_d or strength is selected (16-bit planes may add a
    # narrowing launch to each, the generic width its own passes)
    assert launches >= len(thetas) + (1 if mask & (B(capi.THETA) | B(capi.STRENGTH)) else 0)
    Ref(g, x, dtype).check(got, thetas, mask, kernel)
    return kernel


@pytest.mark.parametrize("dtype", DTYPES)
def test_fallback_forms(dtype):
    # cooperative loader (130 x 131 frames: rows of 524 bytes), a 200-byte input pitch, non-default spacing, width 3
    g = G2Batch()
    k = _fallback_case(g, _frames(2, 130, 131, False), dtype)
    assert "/ldg" in k
    k = _fallback_case(g, _frames(2, 130, 131, True), dtype, mask=capi.G2_MASK_STEER5)
    assert "/ldg-u8" in k
    padded = _frames(2, 96, 50, False)[:, :, :48]
    assert padded.stride(1) * 4 == 200
    _fallback_case(g, padded, dtype)
    _fallback_case(G2Batch(spacing=0.5), _frames(2, 96, 128, False), dtype, mask=B(capi.E) | B(capi.THETA))
    _fallback_case(G2Batch(width=3), _frames(2, 96, 128, False), dtype, mask=B(capi.G2T) | B(capi.STRENGTH))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_layouts(dtype):
    g = G2Batch()
    n, rows, cols, N = 3, 200, 256, 6
    x = _frames(n, rows, cols, False, seed=1)
    thetas = ANGLES[2:2 + N]
    mask = capi.G2_BANK_PLANES
    ref = Ref(g, x, dtype)
    per = [p for p in range(capi.G2_NPLANES) if mask >> p & 1 and p not in ONCE]
    # frame-major: [n, N, rows, cols] storage seen as [N, n, rows, cols]; every plane of a call shares one frame stride, so
    # theta / strength sit in slot 0 of the same kind of storage
    outs = {p: torch.empty((n, N, rows, cols), dtype=dtype, device="cuda").transpose(0, 1) for p in per}
    outs.update({p: torch.empty((n, N, rows, cols), dtype=dtype, device="cuda")[:, 0] for p in ONCE})
    got, launches, kernel = _bank(g, x, thetas, mask, outs=outs, out_dtype=dtype)
    assert kernel.startswith("g2_bank/") and launches == 1
    ref.check(got, thetas, mask, "frame-major")
    # padded pitches (rows of cols + 24 elements)
    outs = {p: torch.empty((N, n, rows, cols + 24), dtype=dtype, device="cuda")[..., :cols] for p in per}
    outs.update({p: torch.empty((n, rows, cols + 24), dtype=dtype, device="cuda")[..., :cols] for p in ONCE})
    got, launches, kernel = _bank(g, x, thetas, mask, outs=outs, out_dtype=dtype)
    assert kernel.startswith("g2_bank/") and launches == 1
    ref.check(got, thetas, mask, "padded")


def test_batch_fields():
    g = G2Batch()
    n, rows, cols = 2, 540, 960
    x = _frames(n, rows, cols, False, seed=2)
    thetas = ANGLES[:8]
    nxt = torch.empty((n, (rows + 1) // 2, (cols + 1) // 2), device="cuda")
    whole, launches, kernel = _bank(g, x, thetas, capi.G2_BANK_PLANES, next_level=nxt)
    assert kernel.startswith("g2_bank/") and launches == 1
    _same(nxt, pyr_down(x), "next_level")
    for dtype in (torch.float32, torch.bfloat16):
        whole = g.steer_bank(x, thetas, capi.G2_BANK_PLANES, out_dtype=dtype)
        for r0, r1 in ((0, 100), (130, 397), (400, rows)):
            part, launches, kernel = _bank(g, x, thetas, capi.G2_BANK_PLANES, band=Band(rows, 0, r0, r1), out_dtype=dtype)
            assert kernel.startswith("g2_bank/") and launches == 1
            for name, t in part.items():
                _same(t, whole[name][..., r0:r1, :], ("band", name, r0, r1))
    # the fallback honours them as well (width 3: the generic path, pyr_down on its own)
    g3 = G2Batch(width=3)
    nxt3 = torch.empty_like(nxt)
    got, _, kernel = _bank(g3, x, thetas[:3], capi.G2_MASK_STEER5, next_level=nxt3)
    assert kernel.startswith("bank-fallback:")
    _same(nxt3, pyr_down(x), "fallback next_level")


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_host_call_matches_device_bank(u8, dtype):
    g = G2Batch()
    n, rows, cols = 7, 64, 128  # 7 frames: chunks of 2, 2, 2 and a short last one of 1
    thetas = ANGLES[3:8]
    mask = capi.G2_BANK_PLANES
    xd = _frames(n, rows, cols, u8, seed=3)
    xh = xd.cpu().pin_memory()
    want = g.steer_bank(xd, thetas, mask, out_dtype=dtype)
    outs = {}
    for p in range(capi.G2_NPLANES):
        if mask >> p & 1:
            shape = (n, rows, cols) if p in ONCE else (len(thetas), n, rows, cols)
            outs[p] = torch.full(shape, float("nan"), dtype=dtype).pin_memory()
    g.steer_bank_host(xh, thetas, mask, outs)
    for p, t in outs.items():
        _same(t, want[capi.G2_PLANE_NAMES[p]].cpu(), ("host", p))
    # frame-major host planes with padded rows
    outs2 = {p: torch.zeros((n, len(thetas), rows, cols + 8), dtype=dtype).pin_memory().transpose(0, 1)[..., :cols]
             for p in outs if p not in ONCE}
    outs2.update({p: torch.zeros((n, len(thetas), rows, cols + 8), dtype=dtype).pin_memory()[:, 0, :, :cols] for p in ONCE})
    g.steer_bank_host(xh, thetas, mask, outs2)
    for p, t in outs2.items():
        _same(t.contiguous(), want[capi.G2_PLANE_NAMES[p]].cpu(), ("host frame-major", p))
