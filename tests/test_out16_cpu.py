"""16-bit output planes (cvs_out_format): argument checks of the *_fmt entry points, which come before any CUDA call (the
handle check included), so an unknown format, a pitch too small or odd for 16-bit planes and a misaligned plane are
argument errors with or without a device.  With a device the buffers are device / host memory the calls may really use
and the accepted geometries run; without one they reach the null-handle / no-device errors, i.e. got past validation."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from cvsteer_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS, COLS = 16, 32


def test_out_format_enum_matches_header():
    txt = open(os.path.join(ROOT, "include", "cvsteer_c.h")).read()
    assert "CVS_OUT_F32 = 0, CVS_OUT_F16 = 1, CVS_OUT_BF16 = 2" in txt
    assert (capi.OUT_F32, capi.OUT_F16, capi.OUT_BF16) == (0, 1, 2)


class _Bufs:
    """Input frame + 20 output planes of ROWS x COLS (room for the odd pitch / offset cases) on the device, or host arrays."""

    def __init__(self, device):
        self.device = device
        if device:
            self.keep = [torch.zeros(ROWS * COLS, device="cuda:0"), torch.zeros((20, ROWS * (COLS + 8)), device="cuda:0")]
            self.inp, self.out = self.keep[0].data_ptr(), self.keep[1].data_ptr()
        else:
            self.keep = [(C.c_float * (ROWS * COLS))(), (C.c_float * (20 * ROWS * (COLS + 8)))()]
            self.inp, self.out = C.addressof(self.keep[0]), C.addressof(self.keep[1])

    def planes(self, offset=0):
        arr = (C.c_void_p * capi.G2_NPLANES)()
        for p in range(capi.G2_NPLANES):
            arr[p] = self.out + p * ROWS * (COLS + 8) * 4 + offset
        return arr


def _batch(bufs, out_pitch):
    b = capi.Batch()
    b.in_, b.in_is_u8, b.n, b.rows, b.cols = bufs.inp, 0, 1, ROWS, COLS
    b.in_pitch, b.in_frame_stride = COLS * 4, COLS * 4 * ROWS
    b.out_pitch, b.out_frame_stride = out_pitch, out_pitch * ROWS
    return b


# (format, out_pitch, plane byte offset, expected words of the error text)
BAD = [(3, COLS * 2, 0, b"out_format"), (-1, COLS * 2, 0, b"out_format"), (capi.OUT_F16, COLS * 2 - 2, 0, b"cols*2"),
       (capi.OUT_BF16, COLS * 2 + 1, 0, b"even out_pitch"), (capi.OUT_F16, COLS * 2, 1, b"2-byte aligned"),
       (capi.OUT_BF16, COLS * 2 + 2, 1, b"2-byte aligned")]


@pytest.mark.parametrize("family", [2, 4])
def test_dev_fmt_arguments_validated_before_any_cuda_call(family):
    lib = capi.lib()
    device = torch.cuda.is_available()
    bufs = _Bufs(device)
    h = C.c_void_p()
    if device:
        capi.check(getattr(lib, f"cvs_g{family}_create")(C.byref(h), 0, 4 if family == 2 else 6, 0.67 if family == 2 else 0.5))
    mask = capi.G2_MASK_FULL if family == 2 else capi.G4_MASK_STEER
    fn = getattr(lib, f"cvs_g{family}_run_batch_dev_fmt")
    try:
        before = lib.cvs_launch_count()
        for fmt, pitch, off, words in BAD:
            rc = fn(h, C.byref(_batch(bufs, pitch)), mask, capi.STEER_DOMINANT, 0.0, None, bufs.planes(off), None, fmt)
            assert rc == capi.ERR_INVALID_ARG and words in lib.cvs_last_error(), (fmt, pitch, off, lib.cvs_last_error())
        assert lib.cvs_launch_count() == before
        # CVS_OUT_F32 through the _fmt call is the fp32 call: a 16-bit pitch is too small for it
        rc = fn(h, C.byref(_batch(bufs, COLS * 2)), mask, capi.STEER_DOMINANT, 0.0, None, bufs.planes(), None, capi.OUT_F32)
        assert rc == capi.ERR_INVALID_ARG and (b"cols*4" in lib.cvs_last_error() or not device), lib.cvs_last_error()
        for fmt in (capi.OUT_F16, capi.OUT_BF16):
            rc = fn(h, C.byref(_batch(bufs, COLS * 2)), mask, capi.STEER_DOMINANT, 0.0, None, bufs.planes(), None, fmt)
            if device:
                assert rc == capi.OK, lib.cvs_last_error()
            else:
                assert rc == capi.ERR_INVALID_ARG and b"handle is null" in lib.cvs_last_error()
        if device:
            torch.cuda.synchronize()
    finally:
        if h.value:
            getattr(lib, f"cvs_g{family}_destroy")(h)


def test_host_fmt_arguments_validated_before_any_cuda_call():
    lib = capi.lib()
    device = torch.cuda.is_available()
    host_in = np.zeros((ROWS, COLS), np.float32)
    host_out = np.zeros((20, ROWS, COLS + 8), np.float16)
    base = host_out.ctypes.data

    def planes(off=0):
        arr = (C.c_void_p * capi.G2_NPLANES)()
        for p in range(capi.G2_NPLANES):
            arr[p] = base + host_out[p].nbytes * p + off
        return arr

    h2, h4 = C.c_void_p(), C.c_void_p()
    if device:
        capi.check(lib.cvs_g2_create(C.byref(h2), 0, 4, 0.67))
        capi.check(lib.cvs_g4_create(C.byref(h4), 0, 6, 0.5))
    inp = C.c_void_p(host_in.ctypes.data)
    calls = {
        "g2": lambda fmt, pitch, off: lib.cvs_g2_run_batch_host_fmt(h2, inp, 1, ROWS, COLS, COLS * 4, COLS * 4 * ROWS, capi.G2_MASK_ORIENT,
                                                                    planes(off), pitch, pitch * ROWS, fmt),
        "g4": lambda fmt, pitch, off: lib.cvs_g4_run_batch_host_fmt(h4, inp, 1, ROWS, COLS, COLS * 4, COLS * 4 * ROWS, capi.G4_MASK_STEER,
                                                                    capi.STEER_SCALAR, 0.3, planes(off), pitch, pitch * ROWS, fmt),
        "multi": lambda fmt, pitch, off: lib.cvs_g2_run_batch_host_multi_fmt(1, None, 4, 0.67, inp, 1, ROWS, COLS, COLS * 4, COLS * 4 * ROWS,
                                                                             capi.G2_MASK_ORIENT, planes(off), pitch, pitch * ROWS, fmt),
    }
    try:
        before = lib.cvs_launch_count()
        for name, call in calls.items():
            for fmt, pitch, off, words in BAD:
                rc = call(fmt, pitch, off)
                assert rc == capi.ERR_INVALID_ARG and words in lib.cvs_last_error(), (name, fmt, pitch, off, lib.cvs_last_error())
        assert lib.cvs_launch_count() == before
        for name, call in calls.items():
            rc = call(capi.OUT_BF16, (COLS + 8) * 2, 0)
            if device:
                assert rc == capi.OK, (name, lib.cvs_last_error())
            elif name == "multi":
                assert rc == capi.ERR_CUDA, lib.cvs_last_error()                 # the per-GPU handle needs a device
            else:
                assert rc == capi.ERR_INVALID_ARG and b"null argument" in lib.cvs_last_error(), lib.cvs_last_error()
    finally:
        for h, fam in ((h2, 2), (h4, 4)):
            if h.value:
                getattr(lib, f"cvs_g{fam}_destroy")(h)


def test_host_planes_share_one_dtype():
    from cvsteer_b200.batch import _host_format
    assert _host_format({capi.E: torch.zeros(2, 2, dtype=torch.bfloat16)}) == (capi.OUT_BF16, 2)
    assert _host_format({capi.E: torch.zeros(2, 2), capi.MAG: torch.zeros(2, 2)}) == (capi.OUT_F32, 4)
    with pytest.raises(capi.CvsError) as e:
        _host_format({capi.E: torch.zeros(2, 2, dtype=torch.float16), capi.MAG: torch.zeros(2, 2)})
    assert e.value.code == capi.ERR_INVALID_ARG
    with pytest.raises(capi.CvsError):
        _host_format({capi.E: torch.zeros(2, 2, dtype=torch.float64)})
