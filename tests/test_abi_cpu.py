"""CPU-only checks of the drop-in boundary: the library loads, exports every symbol include/cvsteer_c.h
declares, generates the reference's taps, and fails loudly (never falls back) without a device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "cvsteer_c.h")).read()
    return sorted(set(re.findall(r"CVS_API\s+[\w\s\*]+?\b(cvs_\w+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from cvsteer_b200 import capi
    lib = capi.lib()
    syms = _header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in cvsteer_c.h but not exported"
    assert sorted(capi.EXPORTED_SYMBOLS) == syms, "ctypes binding and header disagree"
    assert b"sm_100a" in lib.cvs_version()


def test_enum_values_match_header():
    from cvsteer_b200 import capi
    txt = open(os.path.join(ROOT, "include", "cvsteer_c.h")).read()
    assert "CVS_C1 = 7" in txt and "CVS_THETA = 10" in txt and "CVS_G2T = 12" in txt and "CVS_EDGES = 17" in txt
    assert capi.C1 == 7 and capi.THETA == 10 and capi.G2T == 12 and capi.EDGES == 17 and capi.G2_NPLANES == 20
    assert "CVS_H4A = 5" in txt and "CVS_G4T = 11" in txt and capi.H4A == 5 and capi.G4T == 11
    assert capi.G2_MASK_ORIENT == 0x4C00 and capi.G2_MASK_FULL == 0x1FC00


def test_host_taps_equal_oracle_taps(taps_default):
    import cvsteer_b200 as cb
    for i, n in enumerate(("g1", "g2", "g3", "h1", "h2", "h3", "h4")):
        assert np.array_equal(cb.make_taps_g2(i), taps_default[n]), n
    for i, n in enumerate(("g1", "g2", "g3", "g4", "g5", "h1", "h2", "h3", "h4", "h5", "h6")):
        assert np.array_equal(cb.make_taps_g4(i), taps_default["G4_" + n]), n


def test_host_taps_other_widths_equal_oracle():
    import cvsteer_b200 as cb
    from oracle import cvsteer_ref as ref
    g2 = (ref.G21, ref.G22, ref.G23, ref.H21, ref.H22, ref.H23, ref.H24)
    g4 = (ref.G41, ref.G42, ref.G43, ref.G44, ref.G45, ref.H41, ref.H42, ref.H43, ref.H44, ref.H45, ref.H46)
    for w, s in ((3, 0.8), (9, 0.31), (1, 1.0), (32, 0.1)):
        for i, fn in enumerate(g2):
            assert np.array_equal(cb.make_taps_g2(i, w, s), ref.create(w, s, fn)[0]), (w, s, i)
        for i, fn in enumerate(g4):
            assert np.array_equal(cb.make_taps_g4(i, w, s), ref.create(w, s, fn)[0]), (w, s, i)


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    import cvsteer_b200 as cb
    from cvsteer_b200 import capi
    with pytest.raises(capi.CvsError) as e:
        cb.SteerableFiltersG2(np.zeros((8, 8), np.float32))
    assert e.value.code == capi.ERR_CUDA
    n = C.c_int(-1)
    assert capi.lib().cvs_device_count(C.byref(n)) == capi.ERR_CUDA


def test_product_code_never_imports_oracle():
    """The shipped package must not reference oracle/ (or cv2) anywhere."""
    pkg = os.path.join(ROOT, "cvsteer_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dp, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn
                assert "import cv2" not in src, fn


def test_header_is_plain_c_and_c_caller_runs():
    """include/cvsteer_c.h compiles as pedantic C99 and a C program can call the library (on this CPU box it reaches the
    no-device error path; on the GPU box tests/test_cpp_dropin_gpu.py runs the same binary against the device)."""
    import subprocess
    subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "cpp"), "abi_c_check"], check=True, capture_output=True)
    r = subprocess.run([os.path.join(ROOT, "tests", "cpp", "abi_c_check")], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)


def test_band_contract_is_validated_before_any_cuda_call():
    """Band mode: the buffer must hold the footprint of the requested output rows; a short halo is an argument error
    (it would silently filter zeros), reported before the library touches CUDA.  An accepted geometry then runs on the
    device (device buffers) or, without one, reaches the no-device error (host buffers: nothing is launched)."""
    import ctypes as C

    import torch

    from cvsteer_b200 import capi
    lib = capi.lib()
    device = torch.cuda.is_available()
    if device:
        keep = torch.zeros(40 * 16, device="cuda:0"), torch.zeros(50 * 8, device="cuda:0")
        buf, out = keep[0].data_ptr(), keep[1].data_ptr()
    else:
        keep = (C.c_float * (40 * 16))(), (C.c_float * (50 * 8))()
        buf, out = C.addressof(keep[0]), C.addressof(keep[1])
    b = capi.Batch()
    b.in_, b.in_is_u8, b.n, b.rows, b.cols = buf, 0, 1, 40, 16
    b.in_pitch, b.in_frame_stride, b.out_pitch, b.out_frame_stride = 64, 64 * 40, 32, 32 * 50
    b.full_rows, b.y_origin, b.out_row_origin = 100, 10, 6                    # buffer = image rows [10, 50)
    for begin, end, ok in ((6, 20, True), (5, 20, False), (6, 26, False), (6, 24, True), (20, 20, False)):
        b.out_row_begin, b.out_row_end = begin, end                          # pyr_down rows y read input rows 2y-2 .. 2y+2
        rc = lib.cvs_pyr_down_dev(0, C.byref(b), out, None)
        if ok:
            assert rc == (capi.OK if device else capi.ERR_CUDA), lib.cvs_last_error()   # geometry accepted
        else:
            assert rc == capi.ERR_INVALID_ARG and (b"need" in lib.cvs_last_error() or b"invalid" in lib.cvs_last_error())
    if device:
        torch.cuda.synchronize()


def test_band_context_arguments_and_no_device():
    """cvs_bands_create validates its arguments before touching CUDA and, without a device, fails loudly (no fallback);
    cvs_plan_bands (host-only) agrees with the Python planner the gloo tests exercise."""
    import torch

    from cvsteer_b200 import capi, multi
    lib = capi.lib()
    h = C.c_void_p()
    for args in ((0, 3, 2, 0, 100, 64, 5), (0, 0, 2, 5, 100, 64, 5), (0, 0, 1, 0, 0, 64, 5), (0, 0, 1, 0, 100, 64, 0)):
        assert lib.cvs_bands_create(C.byref(h), *args, capi.G2_MASK_ORIENT, 4, 0.67) == capi.ERR_INVALID_ARG, args
    assert lib.cvs_bands_create(C.byref(h), 0, 0, 1, 0, 100, 64, 5, 0, 4, 0.67) == capi.ERR_INVALID_ARG      # empty mask
    if not torch.cuda.is_available():
        assert lib.cvs_bands_create(C.byref(h), 0, 0, 1, 0, 100, 64, 5, capi.G2_MASK_ORIENT, 4, 0.67) == capi.ERR_CUDA
        assert not h.value
    for rows, world, levels in ((1000, 3, 5), (32768, 8, 5), (77, 4, 3), (16, 8, 5)):
        plan = (C.c_int * (world * levels * 4))()
        rpl = (C.c_int * levels)()
        assert lib.cvs_plan_bands(rows, world, levels, 4, plan, rpl) == 0
        py = multi.plan_bands(rows, world, levels)
        for r in range(world):
            for l in range(levels):
                q = plan[(r * levels + l) * 4:(r * levels + l) * 4 + 4]
                assert (q[0], q[1]) == py[r].out[l] and (q[2], q[3]) == py[r].have[l], (rows, world, r, l)
        assert list(rpl) == py[0].rows
