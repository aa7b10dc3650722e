"""Device-resident batch + pyramid path over torch CUDA tensors.

torch is plumbing here: it owns device memory and streams; every kernel launched is ours, through the C ABI
(cvs_g2_run_batch_dev / cvs_g4_run_batch_dev / cvs_pyr_down_dev).  This is the reference's per-file loop
(example/steer.cpp:69-124) with the file I/O removed: frames in HBM in, selected planes in HBM out.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import torch

from . import capi


@dataclass
class Band:
    """Row band of one tall image (SURVEY section 8e): the input tensor holds image rows
    [y_origin, y_origin + tensor_rows) of an image `full_rows` tall; outputs are produced for image rows
    [row_begin, row_end) and land at row (y - row_begin) of the output tensors."""
    full_rows: int
    y_origin: int
    row_begin: int
    row_end: int


def _as_batch(x: torch.Tensor) -> torch.Tensor:
    if x.dim() == 2:
        x = x.unsqueeze(0)
    if x.dim() != 3 or not x.is_cuda or x.dtype not in (torch.float32, torch.uint8):
        raise capi.CvsError(capi.ERR_INVALID_ARG, "frames must be a CUDA tensor [n, rows, cols] of float32 or uint8")
    if x.stride(2) != 1:
        x = x.contiguous()
    return x


def _batch_struct(x: torch.Tensor, out_pitch: int, out_frame_stride: int, band: Optional[Band]) -> capi.Batch:
    b = capi.Batch()
    es = x.element_size()
    b.in_ = x.data_ptr()
    b.in_is_u8 = int(x.dtype == torch.uint8)
    b.n, b.rows, b.cols = x.shape
    b.in_pitch = x.stride(1) * es
    b.in_frame_stride = x.stride(0) * es if x.shape[0] > 1 else x.stride(1) * es * x.shape[1]
    b.out_pitch, b.out_frame_stride = out_pitch, out_frame_stride
    if band is not None:
        b.full_rows, b.y_origin = band.full_rows, band.y_origin
        b.out_row_begin, b.out_row_end, b.out_row_origin = band.row_begin, band.row_end, band.row_begin
    return b


# output plane dtype -> cvs_out_format: 16-bit planes are the fp32 planes rounded to nearest even (include/cvsteer_c.h)
_OUT_FORMATS = {torch.float32: capi.OUT_F32, torch.float16: capi.OUT_F16, torch.bfloat16: capi.OUT_BF16}


def _out_format(dtype) -> int:
    if dtype not in _OUT_FORMATS:
        raise capi.CvsError(capi.ERR_INVALID_ARG, f"output planes are float32, float16 or bfloat16, not {dtype}")
    return _OUT_FORMATS[dtype]


def _host_format(outs_host: Dict[int, torch.Tensor]):
    """(cvs_out_format, element size) of the pinned output planes of one run_host call: they share one dtype."""
    dtypes = {t.dtype for t in outs_host.values()}
    if len(dtypes) != 1:
        raise capi.CvsError(capi.ERR_INVALID_ARG, f"the output planes of one call share one dtype, got {sorted(map(str, dtypes))}")
    dt = dtypes.pop()
    return _out_format(dt), torch.empty((), dtype=dt).element_size()


def _host_frames(x: torch.Tensor):
    """(8-bit?, row step, frame step in bytes) of the host frames of one run_host call: float32 or uint8, rows of unit stride.
    Checked here because the C calls take raw pointers and steps: any other layout would be read as the wrong bytes."""
    if x.is_cuda or x.dtype not in (torch.float32, torch.uint8):
        raise capi.CvsError(capi.ERR_INVALID_ARG, f"host frames are a CPU tensor of float32 or uint8, not {x.dtype} on {x.device}")
    if x.stride(-1) != 1:
        raise capi.CvsError(capi.ERR_INVALID_ARG, f"host frames need rows of unit stride, got strides {tuple(x.stride())}")
    es = x.element_size()
    return x.dtype == torch.uint8, x.stride(1) * es, x.stride(0) * es


def _bank_angles(thetas, mask: int, bank_planes: int):
    """float array of the bank's angles; the angle count and the mask (bits of the family's bank planes) checked before
    anything touches a device."""
    th = [float(t) for t in thetas]
    if not 1 <= len(th) <= capi.BANK_MAX_ANGLES:
        raise capi.CvsError(capi.ERR_INVALID_ARG, f"a bank steers to 1..{capi.BANK_MAX_ANGLES} angles, got {len(th)}")
    if not mask or mask & ~bank_planes:
        raise capi.CvsError(capi.ERR_INVALID_ARG, f"bank mask 0x{mask:x}: bank planes are 0x{bank_planes:x}")
    return (C.c_float * len(th))(*th)


def _bank_layout(outs: Dict[int, torch.Tensor], planes, shape_angle, shape_once, per_angle_mask: int):
    """(out_pitch, out_frame_stride, angle_stride) in bytes shared by the bank's planes: per-angle planes (bits of
    per_angle_mask) are [N, n, rows, cols] views, G2's theta / strength [n, rows, cols]; any strides with unit column stride."""
    lay = set()
    for p in planes:
        t = outs[p]
        per_angle = per_angle_mask >> p & 1
        want = shape_angle if per_angle else shape_once
        if tuple(t.shape) != want or t.stride(-1) != 1:
            raise capi.CvsError(capi.ERR_SIZE_MISMATCH, f"output plane {p}: need {want} with unit column stride, got {tuple(t.shape)}")
        es = t.element_size()
        st = [s * es for s in t.stride()]
        lay.add((st[-2], st[-3], st[0] if per_angle else None))
    pitches = {l[:2] for l in lay}
    angle = {l[2] for l in lay if l[2] is not None}
    if len(pitches) != 1 or len(angle) > 1:
        raise capi.CvsError(capi.ERR_INVALID_ARG, "the bank's planes share one row pitch and frame stride, and the per-angle "
                                                  "planes one angle stride")
    pitch, fstride = pitches.pop()
    return pitch, fstride, angle.pop() if angle else 0


def _stream_ptr(stream):
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


class _FusedBatch:
    _prefix = ""
    _names: Sequence[str] = ()
    _bank_planes = 0      # mask bits a steering bank takes
    _bank_per_angle = 0   # ... those of them written once per angle

    def __init__(self, width: int, spacing: float, device: Optional[int] = None):
        self._lib = capi.lib()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self._h = C.c_void_p()
        capi.check(getattr(self._lib, f"cvs_{self._prefix}_create")(C.byref(self._h), self.device, width, spacing))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            getattr(self._lib, f"cvs_{self._prefix}_destroy")(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self, frames: torch.Tensor, mask: int, steer: int = capi.STEER_DOMINANT, theta: float = 0.0,
            theta_map: Optional[torch.Tensor] = None, outs: Optional[Dict[int, torch.Tensor]] = None,
            band: Optional[Band] = None, stream=None, next_level: Optional[torch.Tensor] = None,
            out_dtype: torch.dtype = torch.float32) -> Dict[str, torch.Tensor]:
        """One fused launch over the whole batch.  Returns {plane name: tensor [n, out_rows, cols]}.
        next_level: optional contiguous float32 [n, (rows+1)//2, (cols+1)//2]; the same launch fills it with
        cv::pyrDown(frames) from the tile it stages anyway (whole frames only).
        out_dtype: float32, or float16 / bfloat16 planes that are the float32 planes rounded to nearest even (theta_map and
        next_level stay float32)."""
        x = _as_batch(frames)
        if x.device.index != self.device:
            raise capi.CvsError(capi.ERR_INVALID_ARG, f"frames live on cuda:{x.device.index}, this handle on cuda:{self.device}")
        n, rows, cols = x.shape
        out_rows = rows if band is None else band.row_end - band.row_begin
        nplanes = len(self._names)
        planes = [p for p in range(nplanes) if mask >> p & 1]
        fmt = _out_format(out_dtype)
        es = 4 if fmt == capi.OUT_F32 else 2
        if outs is None:
            outs = {p: torch.empty((n, out_rows, cols), dtype=out_dtype, device=x.device) for p in planes}
        arr = (C.c_void_p * nplanes)()
        for p in planes:
            t = outs[p]
            if t.shape != (n, out_rows, cols) or t.dtype != out_dtype or not t.is_contiguous() or not t.is_cuda:
                raise capi.CvsError(capi.ERR_SIZE_MISMATCH, f"output plane {p}: need contiguous CUDA {out_dtype} {(n, out_rows, cols)}")
            arr[p] = t.data_ptr()
        tm = None
        if steer == capi.STEER_MAP:
            # the kernel reads theta_map + frame * out_frame_stride: the map needs the full [n, out_rows, cols] extent
            if theta_map is not None and theta_map.dim() == 2 and n == 1:
                theta_map = theta_map.unsqueeze(0)
            if (theta_map is None or tuple(theta_map.shape) != (n, out_rows, cols) or theta_map.dtype != torch.float32
                    or not theta_map.is_contiguous() or theta_map.device != x.device):
                raise capi.CvsError(capi.ERR_SIZE_MISMATCH,
                                    f"theta_map must be a contiguous float32 tensor {(n, out_rows, cols)} on {x.device}")
            tm = C.c_void_p(theta_map.data_ptr())
        b = _batch_struct(x, cols * es, out_rows * cols * es, band)
        if next_level is not None:
            want = (n, (rows + 1) // 2, (cols + 1) // 2)
            if tuple(next_level.shape) != want or next_level.dtype != torch.float32 or not next_level.is_contiguous():
                raise capi.CvsError(capi.ERR_SIZE_MISMATCH, f"next_level must be contiguous float32 {want}")
            b.next_level = next_level.data_ptr()
            b.next_pitch, b.next_frame_stride = want[2] * 4, want[1] * want[2] * 4
        with torch.cuda.device(self.device):   # the C call makes the handle's GPU current; torch's current device is restored
            if fmt == capi.OUT_F32:
                fn = getattr(self._lib, f"cvs_{self._prefix}_run_batch_dev")
                capi.check(fn(self._h, C.byref(b), mask, steer, theta, tm, arr, _stream_ptr(stream)))
            else:
                fn = getattr(self._lib, f"cvs_{self._prefix}_run_batch_dev_fmt")
                capi.check(fn(self._h, C.byref(b), mask, steer, theta, tm, arr, _stream_ptr(stream), fmt))
        return {self._names[p]: outs[p] for p in planes}

    def run_pyramid(self, frames: torch.Tensor, levels: int, mask: int, **kw) -> List[Dict[str, torch.Tensor]]:
        """Every pyramid level stays resident on the device: level l+1 = pyr_down(level l), then one fused
        launch per level (config 3 of BASELINE.json).  Keyword arguments go to run(), out_dtype included; the levels
        themselves (the next level's input) stay float32."""
        res, cur = [], _as_batch(frames)
        fuse = kw.pop("fuse_pyramid", True)
        for l in range(levels):
            nxt = None
            if l + 1 < levels and fuse:
                n, r, c = cur.shape
                nxt = torch.empty((n, (r + 1) // 2, (c + 1) // 2), dtype=torch.float32, device=cur.device)
            res.append(self.run(cur, mask, next_level=nxt, **kw))
            if l + 1 < levels:
                cur = nxt if fuse else pyr_down(cur, stream=kw.get("stream"))
        return res

    def steer_bank(self, frames: torch.Tensor, thetas, mask: Optional[int] = None, outs: Optional[Dict[int, torch.Tensor]] = None,
                   out_dtype: torch.dtype = torch.float32, band: Optional[Band] = None, next_level: Optional[torch.Tensor] = None,
                   stream=None) -> Dict[str, torch.Tensor]:
        """Steering bank (cvs_g2_steer_bank_dev / cvs_g4_steer_bank_dev): one filtering pass, then the planes of `mask` (default:
        every per-angle plane of the family) at every angle of `thetas` (1..16 of them).  Returns {name: tensor}:
        [N, n, out_rows, cols] for the per-angle planes (G2: g2, h2, e, magnitude, phase; G4: g4, h4, magnitude, phase),
        [n, out_rows, cols] for G2's theta and strength.  Each per-angle plane k is, bit for bit, that plane of
        run(frames, G2_MASK_STEER5 / G4_MASK_STEER, STEER_SCALAR, thetas[k]) -- for G4 on uint8 frames, of that call on
        frames.float() -- and G2's theta / strength those of run(frames, G2_MASK_ORIENT).
        outs: optional {plane: tensor} of those shapes with any strides of unit column stride, e.g. a [n, N, rows, cols]
        tensor seen through .transpose(0, 1); the planes share one row pitch and frame stride.  band and next_level as in run()."""
        mask = self._bank_per_angle if mask is None else mask
        th = _bank_angles(thetas, mask, self._bank_planes)
        x = _as_batch(frames)
        if x.device.index != self.device:
            raise capi.CvsError(capi.ERR_INVALID_ARG, f"frames live on cuda:{x.device.index}, this handle on cuda:{self.device}")
        n, rows, cols = x.shape
        out_rows = rows if band is None else band.row_end - band.row_begin
        nplanes = len(self._names)
        planes = [p for p in range(nplanes) if mask >> p & 1]
        fmt = _out_format(out_dtype)
        shape_angle, shape_once = (len(th), n, out_rows, cols), (n, out_rows, cols)
        if outs is None:
            outs = {p: torch.empty(shape_angle if self._bank_per_angle >> p & 1 else shape_once, dtype=out_dtype, device=x.device)
                    for p in planes}
        for p in planes:
            if p not in outs:
                raise capi.CvsError(capi.ERR_INVALID_ARG, f"no output plane for {p}")
            if outs[p].dtype != out_dtype or outs[p].device != x.device:
                raise capi.CvsError(capi.ERR_SIZE_MISMATCH, f"output plane {p}: need {out_dtype} on {x.device}")
        pitch, fstride, astride = _bank_layout(outs, planes, shape_angle, shape_once, self._bank_per_angle)
        arr = (C.c_void_p * nplanes)()
        for p in planes:
            arr[p] = outs[p].data_ptr()
        b = _batch_struct(x, pitch, fstride, band)
        if next_level is not None:
            want = (n, (rows + 1) // 2, (cols + 1) // 2)
            if tuple(next_level.shape) != want or next_level.dtype != torch.float32 or not next_level.is_contiguous():
                raise capi.CvsError(capi.ERR_SIZE_MISMATCH, f"next_level must be contiguous float32 {want}")
            b.next_level = next_level.data_ptr()
            b.next_pitch, b.next_frame_stride = want[2] * 4, want[1] * want[2] * 4
        with torch.cuda.device(self.device):
            fn = getattr(self._lib, f"cvs_{self._prefix}_steer_bank_dev")
            capi.check(fn(self._h, C.byref(b), th, len(th), mask, arr, astride, _stream_ptr(stream), fmt))
        return {self._names[p]: outs[p] for p in planes}

    def steer_bank_host(self, frames_host: torch.Tensor, thetas, mask: int, outs_host: Dict[int, torch.Tensor]):
        """Host-buffer twin of steer_bank (cvs_g2_steer_bank_host / cvs_g4_steer_bank_host): pinned float32 or uint8 frames
        [n, rows, cols] in, pinned planes out ([N, n, rows, cols] per angle, [n, rows, cols] for G2's theta / strength, one
        dtype that selects the format)."""
        th = _bank_angles(thetas, mask, self._bank_planes)
        x = frames_host
        u8, step, fstride = _host_frames(x)
        n, rows, cols = x.shape
        fmt, _ = _host_format(outs_host)
        nplanes = len(self._names)
        planes = [p for p in range(nplanes) if mask >> p & 1]
        missing = [p for p in planes if p not in outs_host]
        if missing:
            raise capi.CvsError(capi.ERR_INVALID_ARG, f"no output plane for {missing}")
        pitch, ofs, astride = _bank_layout(outs_host, planes, (len(th), n, rows, cols), (n, rows, cols), self._bank_per_angle)
        arr = (C.c_void_p * nplanes)()
        for p in planes:
            arr[p] = outs_host[p].data_ptr()
        fn = getattr(self._lib, f"cvs_{self._prefix}_steer_bank_host")
        capi.check(fn(self._h, C.c_void_p(x.data_ptr()), int(u8), n, rows, cols, step, fstride, th, len(th), mask, arr, pitch, ofs, astride,
                      fmt))

    def last_launch(self):
        g = (C.c_int * 3)()
        blk, sm = C.c_int(), C.c_int()
        name = C.create_string_buffer(96)
        capi.check(self._lib.cvs_g2_last_launch(self._h, g, C.byref(blk), C.byref(sm), name, 96))
        return {"grid": list(g), "block": blk.value, "smem": sm.value, "kernel": name.value.decode()}


class G2Batch(_FusedBatch):
    _prefix = "g2"
    _names = capi.G2_PLANE_NAMES
    _bank_planes = capi.G2_BANK_PLANES
    _bank_per_angle = capi.G2_MASK_STEER5

    def __init__(self, width: int = 4, spacing: float = 0.67, device: Optional[int] = None):
        super().__init__(width, spacing, device)

    def run_host(self, frames_host: torch.Tensor, mask: int, outs_host: Dict[int, torch.Tensor]):
        """End-to-end host-buffer call (cvs_g2_run_batch_host): pinned host frames in, pinned host planes out.  The
        planes' dtype (float32, float16 or bfloat16, the same for all) selects the output format.  uint8 frames go up as
        bytes (cvs_g2_run_batch_host_u8) and give the planes of the same frames as float32."""
        x = frames_host
        n, rows, cols = x.shape
        u8, step, fstride = _host_frames(x)
        fmt, es = _host_format(outs_host)
        arr = (C.c_void_p * capi.G2_NPLANES)()
        for p, t in outs_host.items():
            arr[p] = t.data_ptr()
        any_out = next(iter(outs_host.values()))
        args = (self._h, C.c_void_p(x.data_ptr()), n, rows, cols, step, fstride, mask, arr,
                any_out.stride(1) * es, any_out.stride(0) * es)
        if u8:
            capi.check(self._lib.cvs_g2_run_batch_host_u8(*args, fmt))
        elif fmt == capi.OUT_F32:
            capi.check(self._lib.cvs_g2_run_batch_host(*args))
        else:
            capi.check(self._lib.cvs_g2_run_batch_host_fmt(*args, fmt))


class G4Batch(_FusedBatch):
    _prefix = "g4"
    _names = capi.G4_PLANE_NAMES
    _bank_planes = capi.G4_BANK_PLANES
    _bank_per_angle = capi.G4_MASK_STEER

    def __init__(self, width: int = 6, spacing: float = 0.5, device: Optional[int] = None):
        super().__init__(width, spacing, device)

    def run_host(self, frames_host: torch.Tensor, mask: int, outs_host: Dict[int, torch.Tensor],
                 theta: Optional[float] = None):
        """End-to-end host-buffer call (cvs_g4_run_batch_host).  theta=None steers at the G4 theta_d.  The planes' dtype
        (float32, float16 or bfloat16, the same for all) selects the output format; uint8 frames as in G2Batch.run_host."""
        x = frames_host
        n, rows, cols = x.shape
        u8, step, fstride = _host_frames(x)
        fmt, es = _host_format(outs_host)
        arr = (C.c_void_p * capi.G4_NPLANES)()
        for p, t in outs_host.items():
            arr[p] = t.data_ptr()
        any_out = next(iter(outs_host.values()))
        src = capi.STEER_DOMINANT if theta is None else capi.STEER_SCALAR
        args = (self._h, C.c_void_p(x.data_ptr()), n, rows, cols, step, fstride, mask, src,
                float(theta or 0.0), arr, any_out.stride(1) * es, any_out.stride(0) * es)
        if u8:
            capi.check(self._lib.cvs_g4_run_batch_host_u8(*args, fmt))
        elif fmt == capi.OUT_F32:
            capi.check(self._lib.cvs_g4_run_batch_host(*args))
        else:
            capi.check(self._lib.cvs_g4_run_batch_host_fmt(*args, fmt))


def pyr_down(frames: torch.Tensor, band: Optional[Band] = None, out_rows: Optional[range] = None,
             stream=None) -> torch.Tensor:
    """cv::pyrDown semantics on a device batch.  With `band`, `frames` holds rows [y_origin, ...) of the input
    level and `band.row_begin/row_end` are rows of the OUTPUT level."""
    x = _as_batch(frames)
    n, rows, cols = x.shape
    oc = (cols + 1) // 2
    orows = (rows + 1) // 2 if band is None else band.row_end - band.row_begin
    out = torch.empty((n, orows, oc), dtype=torch.float32, device=x.device)
    b = _batch_struct(x, oc * 4, orows * oc * 4, band)
    capi.check(capi.lib().cvs_pyr_down_dev(x.device.index or 0, C.byref(b), C.c_void_p(out.data_ptr()),
                                           _stream_ptr(stream)))
    return out


def ffma_peak(form: int = 2, iters: int = 20000, device: int = 0):
    """Measured FP32 FFMA issue rate (instr/s) for the roofline denominator."""
    v, ms = C.c_double(), C.c_float()
    capi.check(capi.lib().cvs_bench_ffma(device, form, iters, C.byref(v), C.byref(ms)))
    return v.value, ms.value
