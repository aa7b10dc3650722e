"""8-bit host frames (cvs_g2/g4_run_batch_host_u8, cvs_g2_run_batch_host_multi_u8): a null `in`, an in_step below cols and the
16-bit output layout errors are argument errors before the handle is looked at and before any CUDA call, with or without a
device.  With a device the buffers are host memory the calls may really use and the accepted geometries run; without one
they reach the null-handle / no-device errors, i.e. got past validation.  run_host's own frame checks need no device."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from cvsteer_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS, COLS = 16, 32
NEW = ("cvs_g2_run_batch_host_u8", "cvs_g4_run_batch_host_u8", "cvs_g2_run_batch_host_multi_u8")

# (null in?, in_step, out_format, out_step, out_frame_stride, expected words of the error text)
BAD = [(True, COLS, capi.OUT_F16, COLS * 2, COLS * 2 * ROWS, b"in is null"),
       (False, COLS - 1, capi.OUT_F16, COLS * 2, COLS * 2 * ROWS, b"in_step"),
       (False, COLS, 3, COLS * 2, COLS * 2 * ROWS, b"out_format"),
       (False, COLS, -1, COLS * 4, COLS * 4 * ROWS, b"out_format"),
       (False, COLS, capi.OUT_BF16, COLS * 2 + 1, (COLS * 2 + 1) * ROWS + 1, b"even out_pitch"),
       (False, COLS, capi.OUT_F16, COLS * 2 - 2, (COLS * 2 - 2) * ROWS, b"cols*2"),
       (False, COLS, capi.OUT_BF16, COLS * 2, COLS * 2 * ROWS + 1, b"even out_frame_stride")]


def test_new_entry_points_are_declared_and_exported():
    txt = open(os.path.join(ROOT, "include", "cvsteer_c.h")).read()
    lib = capi.lib()
    for name in NEW:
        assert f"CVS_API int {name}(" in txt and name in capi.EXPORTED_SYMBOLS
        getattr(lib, name)


def test_host_u8_arguments_validated_before_any_cuda_call():
    lib = capi.lib()
    device = torch.cuda.is_available()
    host_in = np.zeros((ROWS, COLS + 8), np.uint8)
    host_out = np.zeros((20, ROWS, COLS + 8), np.float32)

    def planes():
        arr = (C.c_void_p * capi.G2_NPLANES)()
        for p in range(capi.G2_NPLANES):
            arr[p] = host_out[p].ctypes.data
        return arr

    h2, h4 = C.c_void_p(), C.c_void_p()
    if device:
        capi.check(lib.cvs_g2_create(C.byref(h2), 0, 4, 0.67))
        capi.check(lib.cvs_g4_create(C.byref(h4), 0, 6, 0.5))

    def inp(null):
        return None if null else C.c_void_p(host_in.ctypes.data)

    calls = {
        "g2": lambda null, step, fmt, ostep, ofs: lib.cvs_g2_run_batch_host_u8(h2, inp(null), 1, ROWS, COLS, step, step * ROWS,
                                                                               capi.G2_MASK_ORIENT, planes(), ostep, ofs, fmt),
        "g4": lambda null, step, fmt, ostep, ofs: lib.cvs_g4_run_batch_host_u8(h4, inp(null), 1, ROWS, COLS, step, step * ROWS,
                                                                               capi.G4_MASK_STEER, capi.STEER_SCALAR, 0.3, planes(),
                                                                               ostep, ofs, fmt),
        "multi": lambda null, step, fmt, ostep, ofs: lib.cvs_g2_run_batch_host_multi_u8(1, None, 4, 0.67, inp(null), 1, ROWS, COLS, step,
                                                                                        step * ROWS, capi.G2_MASK_ORIENT, planes(), ostep,
                                                                                        ofs, fmt),
    }
    try:
        before = lib.cvs_launch_count()
        for name, call in calls.items():
            for null, step, fmt, ostep, ofs, words in BAD:
                rc = call(null, step, fmt, ostep, ofs)
                assert rc == capi.ERR_INVALID_ARG and words in lib.cvs_last_error(), (name, words, lib.cvs_last_error())
        assert lib.cvs_launch_count() == before
        # accepted layouts, fp32 planes included; rows of the 8-bit frames may be padded (in_step > cols)
        for name, call in calls.items():
            for fmt, es in ((capi.OUT_F32, 4), (capi.OUT_F16, 2)):
                rc = call(False, COLS + 8, fmt, (COLS + 8) * es, (COLS + 8) * es * ROWS)
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


def test_host_frames_layout():
    from cvsteer_b200.batch import _host_frames
    assert _host_frames(torch.zeros((3, 4, 5), dtype=torch.uint8)) == (True, 5, 20)
    assert _host_frames(torch.zeros((3, 4, 8))[:, :, :5]) == (False, 32, 128)
    for x in (torch.zeros((3, 4, 5), dtype=torch.float64), torch.zeros((3, 4, 5), dtype=torch.int16),
              torch.zeros((3, 4, 5), dtype=torch.float16), torch.zeros((3, 5, 4), dtype=torch.uint8).transpose(1, 2)):
        with pytest.raises(capi.CvsError) as e:
            _host_frames(x)
        assert e.value.code == capi.ERR_INVALID_ARG
