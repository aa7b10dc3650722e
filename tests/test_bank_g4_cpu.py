"""G4/H4 steering banks (cvs_g4_steer_bank_dev / _host, G4Batch.steer_bank / steer_bank_host): every argument error is
CVS_ERR_INVALID_ARG before the handle is looked at and before any CUDA call, with or without a device.  The calls get a null
handle, so an accepted argument set reaches the handle check ("handle" / "null argument" in the error) and nothing runs."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from cvsteer_b200 import capi
from cvsteer_b200.batch import G2Batch, G4Batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_FR, ROWS, COLS = 2, 16, 32
PLANE = ROWS * COLS * 4  # one dense fp32 plane
B = capi.bit

HOST = np.zeros(4 << 20, np.uint8)  # stands in for every buffer: nothing may be read or written


def _planes(null=(), n=capi.G4_NPLANES):
    arr = (C.c_void_p * n)()
    for p in range(n):
        arr[p] = None if p in null else HOST.ctypes.data
    return arr


def _thetas(k):
    return (C.c_float * max(k, 1))(*([0.25] * max(k, 1)))


GOOD = dict(k=4, null_th=False, mask=capi.G4_MASK_STEER, null=(), fmt=capi.OUT_F32, pitch=COLS * 4, fs=PLANE, ast=N_FR * PLANE)
BAD = [
    (dict(k=0), b"n_angles"),
    (dict(k=17), b"n_angles"),
    (dict(null_th=True), b"thetas is null"),
    # no theta_d / strength and no basis planes in a G4 bank
    (dict(mask=capi.G4_MASK_STEER | B(capi.G4_THETA)), b"mask"),
    (dict(mask=B(capi.G4_STRENGTH)), b"mask"),
    (dict(mask=B(capi.G4A)), b"mask"),
    (dict(mask=capi.G4_MASK_STEER | B(capi.H4F)), b"mask"),
    (dict(mask=B(17)), b"mask"),
    (dict(mask=0), b"mask"),
    (dict(null=(capi.MAG4,)), b"outs[13] is null"),
    (dict(mask=B(capi.H4T), null=(capi.H4T,)), b"outs[12] is null"),
    (dict(fmt=3), b"out_format"),
    (dict(fmt=capi.OUT_F16, pitch=COLS * 2 - 2, fs=PLANE, ast=4 * PLANE), b"cols*2"),
    (dict(fmt=capi.OUT_BF16, pitch=COLS * 2 + 1, fs=PLANE + 16, ast=8 * PLANE), b"even out_pitch"),
    (dict(fmt=capi.OUT_F16, pitch=COLS * 2, fs=PLANE, ast=N_FR * PLANE + 1), b"angle_stride"),
    (dict(pitch=COLS * 4 - 4), b"out_pitch"),
    # overlapping (angle, frame) planes: angle-major with the angles too close, frame-major with the frames too close,
    # a smaller stride below one plane, equal strides
    (dict(ast=PLANE), b"overlap"),
    (dict(fs=4 * PLANE - 4, ast=PLANE), b"overlap"),
    (dict(fs=PLANE - 4), b"overlap"),
    (dict(fs=PLANE, ast=PLANE), b"overlap"),
    (dict(k=1, fs=PLANE - 4), b"overlap"),
]
ACCEPTED = [dict(), dict(fs=4 * PLANE, ast=PLANE), dict(k=1, ast=0), dict(mask=B(capi.G4T) | B(capi.H4T)), dict(mask=B(capi.PHASE4)),
            dict(fmt=capi.OUT_BF16, pitch=COLS * 2, fs=PLANE // 2, ast=N_FR * PLANE // 2), dict(k=16, ast=N_FR * PLANE)]


def _dev_call(lib, a, u8=False, fn="cvs_g4_steer_bank_dev"):
    b = capi.Batch()
    b.in_ = HOST.ctypes.data
    b.in_is_u8 = int(u8)
    b.n, b.rows, b.cols = N_FR, ROWS, COLS
    b.in_pitch, b.in_frame_stride = COLS * 4, PLANE
    b.out_pitch, b.out_frame_stride = a["pitch"], a["fs"]
    return getattr(lib, fn)(None, C.byref(b), None if a["null_th"] else _thetas(a["k"]), a["k"], a["mask"], _planes(a["null"]), a["ast"], None,
                            a["fmt"])


def _host_call(lib, a, in_step=COLS * 4, u8=False):
    return lib.cvs_g4_steer_bank_host(None, HOST.ctypes.data, int(u8), N_FR, ROWS, COLS, in_step, in_step * ROWS,
                                      None if a["null_th"] else _thetas(a["k"]), a["k"], a["mask"], _planes(a["null"]), a["pitch"], a["fs"],
                                      a["ast"], a["fmt"])


def test_g4_bank_symbols_are_declared_and_exported():
    txt = open(os.path.join(ROOT, "include", "cvsteer_c.h")).read()
    for name in ("cvs_g4_steer_bank_dev", "cvs_g4_steer_bank_host"):
        assert f"CVS_API int {name}(" in txt and name in capi.EXPORTED_SYMBOLS
        getattr(capi.lib(), name)
    assert "#define CVS_G4_BANK_PLANES CVS_G4_MASK_STEER" in txt
    assert capi.G4_BANK_PLANES == capi.G4_MASK_STEER == B(capi.G4T) | B(capi.H4T) | B(capi.MAG4) | B(capi.PHASE4) == 0x7800


@pytest.mark.parametrize("entry", ["dev", "host"])
def test_g4_bank_arguments_validated_before_any_cuda_call(entry):
    lib = capi.lib()
    call = _dev_call if entry == "dev" else _host_call
    before = lib.cvs_launch_count()
    for change, words in BAD:
        rc = call(lib, {**GOOD, **change})
        assert rc == capi.ERR_INVALID_ARG and words in lib.cvs_last_error(), (change, words, lib.cvs_last_error())
    for change in ACCEPTED:  # past validation: the null handle is what stops them
        rc = call(lib, {**GOOD, **change})
        assert rc == capi.ERR_INVALID_ARG and (b"handle" in lib.cvs_last_error() or b"null argument" in lib.cvs_last_error()), (
            change, lib.cvs_last_error())
    assert lib.cvs_launch_count() == before


def test_g4_bank_host_in_step_and_null_in():
    lib = capi.lib()
    for u8, step in ((False, COLS * 4 - 4), (True, COLS - 1)):
        assert _host_call(lib, GOOD, in_step=step, u8=u8) == capi.ERR_INVALID_ARG and b"in_step" in lib.cvs_last_error()
    assert _host_call(lib, GOOD, in_step=COLS, u8=True) == capi.ERR_INVALID_ARG and b"null argument" in lib.cvs_last_error()
    rc = lib.cvs_g4_steer_bank_host(None, None, 0, N_FR, ROWS, COLS, COLS * 4, PLANE, _thetas(2), 2, capi.G4_MASK_STEER, _planes(),
                                    COLS * 4, PLANE, N_FR * PLANE, capi.OUT_F32)
    assert rc == capi.ERR_INVALID_ARG and b"in is null" in lib.cvs_last_error()


def test_each_bank_call_checks_its_own_familys_planes():
    lib = capi.lib()
    rc = _dev_call(lib, {**GOOD, "mask": capi.G2_MASK_STEER5})
    assert rc == capi.ERR_INVALID_ARG and b"bank planes are 0x7800" in lib.cvs_last_error()
    rc = _dev_call(lib, {**GOOD, "mask": capi.G4_MASK_STEER | B(capi.G4A)}, fn="cvs_g2_steer_bank_dev")  # bit 0: G2's G2A
    assert rc == capi.ERR_INVALID_ARG and b"bank planes are 0x%x" % capi.G2_BANK_PLANES in lib.cvs_last_error()


def _unbound(cls):
    """A batch whose handle is null: its methods run their own checks, and any C call they reach fails at the handle."""
    g = cls.__new__(cls)
    g._lib, g._h, g.device = capi.lib(), C.c_void_p(), 0
    return g


def test_python_g4_bank_methods_reject_bad_arguments_first():
    g = _unbound(G4Batch)
    frames = torch.zeros((N_FR, ROWS, COLS))
    outs = {p: torch.zeros((4, N_FR, ROWS, COLS)) for p in range(capi.G4_NPLANES) if capi.G4_MASK_STEER >> p & 1}
    bad = [([], capi.G4_MASK_STEER), ([0.1] * 17, capi.G4_MASK_STEER), ([0.1], capi.G4_MASK_STEER | B(capi.G4_THETA)),
           ([0.1], B(capi.G4A)), ([0.1], 0)]
    for thetas, mask in bad:
        for call in (lambda: g.steer_bank(frames, thetas, mask), lambda: g.steer_bank_host(frames, thetas, mask, outs)):
            with pytest.raises(capi.CvsError) as e:
                call()
            assert e.value.code == capi.ERR_INVALID_ARG
    with pytest.raises(capi.CvsError) as e:
        g.steer_bank(frames, [0.1], B(capi.G4_STRENGTH))
    assert "bank planes are 0x7800" in str(e.value)
    # host frames: float16 is neither float32 nor uint8
    with pytest.raises(capi.CvsError) as e:
        g.steer_bank_host(frames.half(), [0.1] * 4, capi.G4_MASK_STEER, outs)
    assert e.value.code == capi.ERR_INVALID_ARG and "float16" in str(e.value)
    # overlapping planes: the angle stride of a [4, n, rows, cols] view over one frame's worth of planes per angle
    packed = torch.zeros((N_FR + 3, ROWS, COLS)).unfold(0, N_FR, 1).permute(0, 3, 1, 2)[:4]
    with pytest.raises(capi.CvsError) as e:
        g.steer_bank_host(frames, [0.1] * 4, B(capi.H4T), {capi.H4T: packed})
    assert e.value.code == capi.ERR_INVALID_ARG and "overlap" in str(e.value)
    # a selected quantity without a tensor
    with pytest.raises(capi.CvsError) as e:
        g.steer_bank_host(frames, [0.1] * 4, capi.G4_MASK_STEER, {p: t for p, t in outs.items() if p != capi.PHASE4})
    assert e.value.code == capi.ERR_INVALID_ARG
    # every G4 bank plane is per angle: a [n, rows, cols] plane is the wrong shape
    with pytest.raises(capi.CvsError) as e:
        g.steer_bank_host(frames, [0.1] * 4, B(capi.G4T), {capi.G4T: torch.zeros((N_FR, ROWS, COLS))})
    assert e.value.code == capi.ERR_SIZE_MISMATCH
    # accepted (default layout, frame-major view): reaches the null handle
    for o in (outs, {p: t.transpose(0, 1).contiguous().transpose(0, 1) for p, t in outs.items()}):
        with pytest.raises(capi.CvsError) as e:
            g.steer_bank_host(frames, [0.1] * 4, capi.G4_MASK_STEER, o)
        assert e.value.code == capi.ERR_INVALID_ARG and "null argument" in str(e.value)


def test_python_bank_methods_keep_each_familys_planes():
    # G2 still defaults to its STEER5 planes and its own messages; G4 to its steered planes
    g2, g4 = _unbound(G2Batch), _unbound(G4Batch)
    with pytest.raises(capi.CvsError) as e:
        g2.steer_bank_host(torch.zeros((N_FR, ROWS, COLS)), [0.1], capi.G4_MASK_STEER | B(capi.G2A), {})
    assert f"bank planes are 0x{capi.G2_BANK_PLANES:x}" in str(e.value)
    for g, planes in ((g2, capi.G2_BANK_PLANES), (g4, capi.G4_BANK_PLANES)):
        assert g._bank_planes == planes
    assert g2._bank_per_angle == capi.G2_MASK_STEER5 and g4._bank_per_angle == capi.G4_MASK_STEER
