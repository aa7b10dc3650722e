"""ctypes binding of libcvsteer_b200.so (include/cvsteer_c.h).

The library is built in-tree by ``cvsteer_b200/csrc/Makefile`` (see ``__graft_entry__.build``).  There is no
fallback of any kind: if the shared library is missing, importing this module raises; if there is no CUDA
device, every compute entry point returns CVS_ERR_CUDA and the wrappers raise :class:`CvsError`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CVS_LIB selects an alternative build of the same library (used to A/B kernel tuning variants on the GPU box)
LIB_PATH = os.environ.get("CVS_LIB") or os.path.join(_HERE, "libcvsteer_b200.so")

# ---- enums (mirror include/cvsteer_c.h) ----
(G2A, G2B, G2C, H2A, H2B, H2C, H2D, C1, C2, C3, THETA, STRENGTH, G2T, H2T, E, MAG, PHASE, EDGES, DARK,
 BRIGHT) = range(20)
G2_NPLANES = 20
G2_PLANE_NAMES = ("g2a", "g2b", "g2c", "h2a", "h2b", "h2c", "h2d", "c1", "c2", "c3", "theta", "strength",
                  "g2", "h2", "e", "magnitude", "phase", "edges", "lines_dark", "lines_bright")
(G4A, G4B, G4C, G4D, G4E, H4A, H4B, H4C, H4D, H4E, H4F, G4T, H4T, MAG4, PHASE4, G4_THETA, G4_STRENGTH) = range(17)
G4_NPLANES = 17
G4_PLANE_NAMES = ("g4a", "g4b", "g4c", "g4d", "g4e", "h4a", "h4b", "h4c", "h4d", "h4e", "h4f", "g4", "h4",
                  "magnitude", "phase", "theta", "strength")


def bit(p):
    return 1 << p


G2_MASK_STATE = 0x00000FFF
G2_MASK_ORIENT = bit(THETA) | bit(STRENGTH) | bit(E)
G2_MASK_FULL = G2_MASK_ORIENT | bit(G2T) | bit(H2T) | bit(MAG) | bit(PHASE)
G2_MASK_LINES = bit(EDGES) | bit(DARK) | bit(BRIGHT)
G2_MASK_STEER5 = bit(G2T) | bit(H2T) | bit(E) | bit(MAG) | bit(PHASE)
G4_MASK_BASIS = 0x000007FF
G4_MASK_STEER = bit(G4T) | bit(H4T) | bit(MAG4) | bit(PHASE4)
G2_BANK_PLANES = G2_MASK_STEER5 | bit(THETA) | bit(STRENGTH)  # per angle: the STEER5 planes; once per pixel: theta, strength
G4_BANK_PLANES = G4_MASK_STEER  # per angle: g4, h4, magnitude, phase (no theta_d / strength: include/cvsteer_c.h)
BANK_MAX_ANGLES = 16
STEER_DOMINANT, STEER_SCALAR, STEER_MAP = 0, 1, 2
OUT_F32, OUT_F16, OUT_BF16 = 0, 1, 2
GATHER_NONE, GATHER_NCCL, GATHER_PEER_STORE, GATHER_PEER_COPY = 0, 1, 2, 3

OK, ERR_INVALID_ARG, ERR_CUDA, ERR_NOT_SETUP, ERR_SIZE_MISMATCH, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5


class Batch(C.Structure):
    _fields_ = [("in_", C.c_void_p), ("in_is_u8", C.c_int), ("n", C.c_int), ("rows", C.c_int), ("cols", C.c_int),
                ("in_pitch", C.c_size_t), ("in_frame_stride", C.c_size_t), ("out_pitch", C.c_size_t),
                ("out_frame_stride", C.c_size_t), ("full_rows", C.c_int), ("y_origin", C.c_int),
                ("out_row_begin", C.c_int), ("out_row_end", C.c_int), ("out_row_origin", C.c_int),
                ("next_level", C.c_void_p), ("next_pitch", C.c_size_t), ("next_frame_stride", C.c_size_t)]


class CvsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cvsteer_b200 error {code}: {msg}")
        self.code = code


# every exported symbol of include/cvsteer_c.h with (restype, argtypes)
_fp = C.POINTER(C.c_float)
_SIGS = {
    "cvs_version": (C.c_char_p, []),
    "cvs_last_error": (C.c_char_p, []),
    "cvs_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "cvs_g2_make_taps": (C.c_int, [C.c_int, C.c_int, C.c_float, _fp]),
    "cvs_g4_make_taps": (C.c_int, [C.c_int, C.c_int, C.c_float, _fp]),
    "cvs_g2_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_float]),
    "cvs_g2_destroy": (C.c_int, [C.c_void_p]),
    "cvs_g2_setup_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "cvs_g2_setup_host_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "cvs_g2_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "cvs_g2_get_plane_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "cvs_g2_steer_scalar_host": (C.c_int, [C.c_void_p, C.c_float] + [C.c_void_p] * 5 + [C.c_size_t]),
    "cvs_g2_steer_map_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t] + [C.c_void_p] * 5 + [C.c_size_t]),
    "cvs_g2_steer_point": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, _fp]),
    "cvs_magnitude_phase_host": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                           C.c_size_t, C.c_int, C.c_int]),
    "cvs_phase_weights_host": (C.c_int, [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                                         C.c_float, C.c_int, C.c_float]),
    "cvs_find_host": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                C.c_int, C.c_int, C.c_float]),
    "cvs_g4_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_float]),
    "cvs_g4_destroy": (C.c_int, [C.c_void_p]),
    "cvs_g4_setup_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "cvs_g4_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "cvs_g4_get_plane_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "cvs_g4_steer_scalar_host": (C.c_int, [C.c_void_p, C.c_float] + [C.c_void_p] * 4 + [C.c_size_t]),
    "cvs_g4_steer_map_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t] + [C.c_void_p] * 4 + [C.c_size_t]),
    "cvs_g2_run_batch_dev": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_uint, C.c_int, C.c_float, C.c_void_p,
                                       C.POINTER(C.c_void_p), C.c_void_p]),
    "cvs_g4_run_batch_dev": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_uint, C.c_int, C.c_float, C.c_void_p,
                                       C.POINTER(C.c_void_p), C.c_void_p]),
    "cvs_g2_run_batch_dev_fmt": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_uint, C.c_int, C.c_float, C.c_void_p,
                                           C.POINTER(C.c_void_p), C.c_void_p, C.c_int]),
    "cvs_g4_run_batch_dev_fmt": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_uint, C.c_int, C.c_float, C.c_void_p,
                                           C.POINTER(C.c_void_p), C.c_void_p, C.c_int]),
    "cvs_pyr_down_dev": (C.c_int, [C.c_int, C.POINTER(Batch), C.c_void_p, C.c_void_p]),
    "cvs_g2_run_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                        C.c_uint, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t]),
    "cvs_plan_bands": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "cvs_enable_peer_access": (C.c_int, [C.c_int, C.c_int]),
    "cvs_shared_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p]),
    "cvs_shared_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    "cvs_shared_close": (C.c_int, [C.c_int, C.c_void_p]),
    "cvs_shared_free": (C.c_int, [C.c_int, C.c_void_p]),
    "cvs_g4_run_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                        C.c_uint, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t]),
    "cvs_g2_run_batch_host_fmt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                            C.c_uint, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_int]),
    "cvs_g4_run_batch_host_fmt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                            C.c_uint, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t,
                                            C.c_int]),
    "cvs_g2_run_batch_host_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                           C.c_uint, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_int]),
    "cvs_g4_run_batch_host_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                           C.c_uint, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t,
                                           C.c_int]),
    "cvs_g2_steer_bank_dev": (C.c_int, [C.c_void_p, C.POINTER(Batch), _fp, C.c_int, C.c_uint, C.POINTER(C.c_void_p), C.c_size_t,
                                        C.c_void_p, C.c_int]),
    "cvs_g2_steer_bank_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, _fp,
                                         C.c_int, C.c_uint, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_size_t, C.c_int]),
    "cvs_g4_steer_bank_dev": (C.c_int, [C.c_void_p, C.POINTER(Batch), _fp, C.c_int, C.c_uint, C.POINTER(C.c_void_p), C.c_size_t,
                                        C.c_void_p, C.c_int]),
    "cvs_g4_steer_bank_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, _fp,
                                         C.c_int, C.c_uint, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_size_t, C.c_int]),
    "cvs_to_u8_dev": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_float, C.c_void_p,
                                C.c_size_t, C.c_size_t, C.c_void_p]),
    "cvs_g2_lines_u8_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]),
    "cvs_g2_run_batch_host_multi": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int,
                                              C.c_int, C.c_size_t, C.c_size_t, C.c_uint, C.POINTER(C.c_void_p), C.c_size_t,
                                              C.c_size_t]),
    "cvs_g2_run_batch_host_multi_fmt": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_float, C.c_void_p, C.c_int,
                                                  C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_uint, C.POINTER(C.c_void_p),
                                                  C.c_size_t, C.c_size_t, C.c_int]),
    "cvs_g2_run_batch_host_multi_u8": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_float, C.c_void_p, C.c_int,
                                                 C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_uint, C.POINTER(C.c_void_p),
                                                 C.c_size_t, C.c_size_t, C.c_int]),
    "cvs_g2_run_bands_host_multi": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int,
                                              C.c_size_t, C.c_int, C.c_uint, C.POINTER(C.POINTER(C.c_void_p)),
                                              C.POINTER(C.c_size_t)]),
    "cvs_bands_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint,
                                   C.c_int, C.c_float]),
    "cvs_bands_destroy": (C.c_int, [C.c_void_p]),
    "cvs_bands_detach": (C.c_int, [C.c_void_p]),
    "cvs_bands_geometry": (C.c_int, [C.c_void_p, C.c_int, C.c_int] + [C.POINTER(C.c_int)] * 6 + [C.POINTER(C.c_size_t)]),
    "cvs_bands_input_dev": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "cvs_bands_upload_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cvs_bands_root_bytes": (C.c_int, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "cvs_bands_root_export": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    "cvs_bands_root_import": (C.c_int, [C.c_void_p, C.c_char_p]),
    "cvs_bands_root_attach": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cvs_bands_root_attach_planes": (C.c_int, [C.c_void_p, C.POINTER(C.POINTER(C.c_void_p)), C.POINTER(C.c_size_t)]),
    "cvs_bands_root_plane": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "cvs_bands_local_plane": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "cvs_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "cvs_bands_nccl_init": (C.c_int, [C.c_void_p, C.c_char_p]),
    "cvs_bands_nccl_attach": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cvs_bands_run": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "cvs_bands_barrier": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cvs_g2_run_bands_dev_multi": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int,
                                             C.c_size_t, C.c_int, C.c_uint, C.c_int, C.POINTER(C.POINTER(C.c_void_p)),
                                             C.POINTER(C.c_size_t)]),
    "cvs_bench_ffma": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), _fp]),
    "cvs_g2_last_launch": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.c_char_p, C.c_int]),
    "cvs_launch_count": (C.c_ulonglong, []),
}
EXPORTED_SYMBOLS = tuple(_SIGS)

_lib = None


def lib():
    """Load the shared library (once).  Raises if it has not been built -- never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C cvsteer_b200/csrc -j` "
                              "(or __graft_entry__.build()); cvsteer_b200 has no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        raise CvsError(rc, lib().cvs_last_error().decode())
    return rc
